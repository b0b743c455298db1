// C-ABI of the B200-native hot path of pseudo_speaker_VAE (see include/psvae_b200.h).
//
// One translation unit: the kernels live in the .cuh files next to this one, this file is the host
// side -- argument checks, workspace carving, tensor-map cache, and the launch sequences that replace
//   VAEModel.forward / decode            (ps_vae/model.py:38-69)
//   PseudoSpeakerVAE.training_step + autograd backward   (ps_vae/lightning.py:67-131)
//   torch.optim.Adam.step                (driven from ps_vae/lightning.py:204-205)
//   unconditional / conditional synthesis (ps_vae/inference.py:10-110)
// Two GEMM engines sit behind every Linear: CUDA-core fp32 (sgemm.cuh, the 1e-5 parity mode) and
// tcgen05/TMEM/TMA bf16 (gemm_tc.cuh, the speed mode).  There is no CPU path.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <map>
#include <utility>
#include <mutex>
#include <tuple>

#include "../../include/psvae_b200.h"
#include "common.cuh"
#include "cosine_topk.cuh"
#include "epilogue.cuh"
#include "gemm_tc.cuh"
#include "decoder_chain.cuh"
#include "kernels.cuh"
#include "langevin.cuh"
#include "philox.cuh"
#include "sgemm.cuh"

namespace psvae {

// ------------------------------------------------------------------------------------------------
// error text, launch counter, options
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[768] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  return (int)e > 0 ? (int)e : 1;
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

struct Options {
  int64_t decode_chunk = 1 << 17;      // rows per pass of psvae_decode (bounds the scratch; measured 347 / 490 / 628 / 696 M samples/s at 16k / 32k / 64k / 128k rows)
  int64_t wgrad_split_cap = 64;        // split-K ceiling of the wgrad GEMMs
  int64_t colsum_rows = 512;           // rows per bias-gradient partial
  int64_t tc_force_bn = 0;             // tests: force the N tile of the tcgen05 engine
  int64_t tc_grid_limit = 0;           // tests: cap the persistent grid
  int64_t tc_two_cta = 1;              // 1: 256-row tiles on CTA pairs (tcgen05 cta_group::2) for BN = 256 shapes
  int64_t langevin_generic = 0;        // tests: force the generic (tile-in-smem) Langevin kernel even where the thread-per-sample one applies
  int64_t fused_head = 1;              // 1 (training, tcgen05 fast mode, latent 64, at most one linear head of <= 4 classes): encoder heads + reparameterisation + KL +
                                       //    classifier forward in ONE kernel (EpiLatent); the classifier's backward then runs inside the latent backward kernel.
                                       //    Measured (round 2, A/B): 0.7867 -> 0.7758 ms/step
  int64_t clf_grad_in_bwd = 0;         // 1 (fast mode, linear-head classifier, also where the fused head does not apply): the fused classifier pass hands only d loss / d logits
                                       //    [B][8] to the backward; d loss / d mu and the classifier's weight / bias gradients are formed by the latent backward kernel.
                                       //    Measured on its own (round 2, A/B): 0.7840 -> 0.7887 ms/step -- slower, so off; the fused head uses the same backward regardless
  int64_t tc_epi_groups = 1;           // 1: thin (K <= 128) BN = 256 forward / dgrad launches use two epilogue groups on alternate tiles (EG2).
                                       //    Measured (round 2, A/B): 0.7832 -> 0.7733 ms/step
  int64_t wgrad_order = 1;             // merged wgrad: 0 = problems in the order the backward pass queued them, 1 = newest first (the gradients written last are
                                       //    still in L2: 0.6826 -> 0.6778 ms/step, A/B round 2), 2 = newest first + batch ranges from the end (same as 1)
  int64_t wgrad_splits = 0;            // experiments: force the number of batch ranges per tile of the merged wgrad (0 = chosen by the launcher: whole rounds of the CTA pairs)
  int64_t tc_bn_rounds = 1;            // 1: a single-tile-column output (N = 256) takes 128 x 128 one-CTA tiles when that fills the rounds of the persistent grid better
                                       //    (dec out + MSE at B = 65,536: 3.46 -> 4 rounds of pair tiles vs 6.92 -> 7 rounds of quarter-size tiles; 0.6502 -> 0.6449 ms/step, A/B)
  int64_t tc_epi_groups_max_k = 128;   // largest contraction length K that still takes the two-epilogue-group kernel
  int64_t tc_merged_wgrad = 1;         // 1 (fast tcgen05 mode): every wgrad of the step runs in ONE persistent launch at the end of the backward pass (gemm_tc_launch_multi_wgrad):
                                       //    the ~8 us fixed cost of a wgrad launch is paid once instead of 8 times
  int64_t decode_chain = 1;            // 1 (tcgen05 mode, two hidden layers <= 512 wide, latent 64, <= 256 outputs, no normalize_decoder): psvae_decode runs the chained
                                       //    decoder kernel (decoder_chain.cuh): z from Philox in-kernel, hidden activations on-chip, one launch for all rows
  int64_t train_chain = 0;             // 1 (training, fast tcgen05 mode, decoder_chain_ok shapes, plain MSE tail, x_hat not requested): the decoder half of the forward pass
                                       //    (dec L0 -> L1 -> last + MSE) runs as ONE chained kernel (decoder_chain.cuh, TRAIN): hidden activations written once, never re-read
  int64_t tc_grouped = 1;              // 1: layers 1..n of the two encoders run as ONE block-diagonal launch each (forward and dgrad) instead of one per encoder
  int64_t pdl = 1;                     // 1: kernels are launched with programmatic stream serialization (their prologue overlaps the predecessor's tail)
  int64_t tc_trace_ptr = 0;            // profiling: device pointer of gridDim.x * 16 cycle counters the GEMM kernels fill (0 = off)
  int64_t tc_trace_skip = 0;           // profiling: with tc_trace_select, tcgen05 launches to let pass before the one that gets the trace buffer
  int64_t tc_trace_select = 0;         // profiling: 1 = only ONE launch is traced (set "tc_trace_skip" = k to pick the (k+1)-th launch from now on)
  int64_t tc_max_stages = 0;           // experiments: cap the depth of the operand ring (0 = what fits)
  int64_t deterministic = 0;           // 1: split-K / bias partials go through ordered two-stage sums instead of TMA reduce-add / atomics
  int64_t topk_key_splits = 0;         // tests: force the number of key ranges per query tile of psvae_cosine_topk (0 = chosen by topk_plan)
};
static Options g_opt;

// ------------------------------------------------------------------------------------------------
// device facts
// ------------------------------------------------------------------------------------------------
struct DevInfo { int checked = 0, ok = 0, sms = 0, major = 0, minor = 0; };
static DevInfo g_dev[64];
static std::mutex g_dev_mu;

static int dev_info(DevInfo** out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("no CUDA device available (%s); this library has no CPU path", cudaGetErrorString(e));
    return -4;
  }
  std::lock_guard<std::mutex> lk(g_dev_mu);
  DevInfo& d = g_dev[dev & 63];
  if (!d.checked) {
    PSVAE_CUDA(cudaDeviceGetAttribute(&d.major, cudaDevAttrComputeCapabilityMajor, dev));
    PSVAE_CUDA(cudaDeviceGetAttribute(&d.minor, cudaDevAttrComputeCapabilityMinor, dev));
    PSVAE_CUDA(cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev));
    d.ok = (d.major == 10);
    d.checked = 1;
  }
  *out = &d;
  return 0;
}
int tc_device_check() {
  DevInfo* d = nullptr;
  PSVAE_TRY(dev_info(&d));
  if (!d->ok) {
    set_error("device is sm_%d%d; this library is built for sm_100a (B200) only and has no fallback", d->major, d->minor);
    return -4;
  }
  return 0;
}
int tc_two_cta() { return (int)g_opt.tc_two_cta; }
int tc_max_stages() { return (int)g_opt.tc_max_stages; }
int tc_epi_groups() { return (int)g_opt.tc_epi_groups; }
int tc_wgrad_splits() { return (int)g_opt.wgrad_splits; }
int tc_bn_rounds() { return (int)g_opt.tc_bn_rounds; }
int tc_epi_groups_max_k() { return (int)g_opt.tc_epi_groups_max_k; }
bool pdl_enabled() { return g_opt.pdl != 0; }
// profiling: the trace buffer goes to ONE launch -- the (tc_trace_skip + 1)-th tcgen05 launch after the option was set (0: every launch, as before)
unsigned long long* tc_trace_ptr() {
  if (!g_opt.tc_trace_ptr) return nullptr;
  if (g_opt.tc_trace_skip < 0) return nullptr;                      // already delivered
  if (g_opt.tc_trace_select) {
    if (g_opt.tc_trace_skip > 0) { --g_opt.tc_trace_skip; return nullptr; }
    g_opt.tc_trace_skip = -1;
  }
  return reinterpret_cast<unsigned long long*>(static_cast<uintptr_t>(g_opt.tc_trace_ptr));
}
int tc_grid_size() {
  DevInfo* d = nullptr;
  if (dev_info(&d) != 0) return PSVAE_NUM_SMS;
  int g = d->sms > 0 ? d->sms : PSVAE_NUM_SMS;
  if (g_opt.tc_grid_limit > 0 && g_opt.tc_grid_limit < g) g = (int)g_opt.tc_grid_limit;
  return g;
}
static int ew_grid(int64_t work_items, int threads = 256) {   // element-wise grid: whole waves of the SM count
  int64_t blocks = ceil_div64(work_items, threads);
  const int64_t cap = (int64_t)PSVAE_NUM_SMS * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ------------------------------------------------------------------------------------------------
// TMA tensor maps (cuTensorMapEncodeTiled through the runtime's driver entry point: no -lcuda needed)
// ------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled g_encode = nullptr;
static std::mutex g_tm_mu;
typedef std::tuple<const void*, int64_t, int64_t, int64_t, int, int> TmKey;
static std::map<TmKey, CUtensorMap> g_tm_cache;

int tc_tensor_map(const TcOperand& op, int64_t K, int box_rows, CUtensorMap* out) {
  std::lock_guard<std::mutex> lk(g_tm_mu);
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    PSVAE_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) {
      set_error("cuTensorMapEncodeTiled not available from this driver");
      return -3;
    }
    g_encode = (PFN_cuTensorMapEncodeTiled)fn;
  }
  const TmKey key(op.ptr, op.rows, op.ld, K, op.mn_major ? 1 : 0, box_rows);
  auto it = g_tm_cache.find(key);
  if (it != g_tm_cache.end()) {
    *out = it->second;
    return 0;
  }
  if ((reinterpret_cast<uintptr_t>(op.ptr) & 15) != 0 || (op.ld % 8) != 0) {
    set_error("tcgen05 operand must be 16-byte aligned with a leading dimension that is a multiple of 8 (ptr=%p ld=%lld)", op.ptr, (long long)op.ld);
    return -2;
  }
  cuuint64_t gdim[2], gstride[1];
  cuuint32_t box[2], estr[2] = {1, 1};
  if (!op.mn_major) {            // row-major [rows][K]: inner = K
    gdim[0] = (cuuint64_t)K; gdim[1] = (cuuint64_t)op.rows;
    box[0] = TC_BK; box[1] = (cuuint32_t)box_rows;
  } else {                       // stored [K][rows]: inner = rows (M or N)
    gdim[0] = (cuuint64_t)op.rows; gdim[1] = (cuuint64_t)K;
    box[0] = 64; box[1] = (cuuint32_t)box_rows;
  }
  gstride[0] = (cuuint64_t)op.ld * sizeof(bf16);
  alignas(64) CUtensorMap tm;
  CUresult r = g_encode(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(op.ptr), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): ptr=%p dims=[%llu,%llu] stride=%llu box=[%u,%u]", (int)r, op.ptr,
              (unsigned long long)gdim[0], (unsigned long long)gdim[1], (unsigned long long)gstride[0], box[0], box[1]);
    return -3;
  }
  if (g_tm_cache.size() > 8192) g_tm_cache.clear();
  g_tm_cache[key] = tm;
  *out = tm;
  return 0;
}

typedef std::tuple<const void*, int, int64_t, int64_t, int64_t, int64_t, int64_t, int> BmKey;
static std::map<BmKey, CUtensorMap> g_bm_cache;

int tc_block_map(const void* ptr, int elem_bytes, int64_t rows, int64_t cols, int64_t ld, int64_t splits, int64_t split_stride, CUtensorMap* out,
                 int box_cols) {
  std::lock_guard<std::mutex> lk(g_tm_mu);
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    PSVAE_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled not available from this driver"); return -3; }
    g_encode = (PFN_cuTensorMapEncodeTiled)fn;
  }
  const BmKey key(ptr, elem_bytes, rows, cols, ld, splits, split_stride, box_cols);
  auto it = g_bm_cache.find(key);
  if (it != g_bm_cache.end()) { *out = it->second; return 0; }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * elem_bytes) % 16 != 0) {
    set_error("tcgen05 epilogue tensors must be 16-byte aligned with 16-byte-multiple row pitch (ptr=%p ld=%lld elem=%d)", ptr, (long long)ld, elem_bytes);
    return -2;
  }
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(splits > 0 ? splits : 1)};
  if (split_stride <= 0) split_stride = rows * ld;
  cuuint64_t gstride[2] = {(cuuint64_t)ld * elem_bytes, (cuuint64_t)split_stride * elem_bytes};
  cuuint32_t box[3] = {(cuuint32_t)box_cols, 32, 1}, estr[3] = {1, 1, 1};
  const int rank = splits > 0 ? 3 : 2;
  alignas(64) CUtensorMap tm;
  CUresult r = g_encode(&tm, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank, const_cast<void*>(ptr), gdim,
                        gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols * elem_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (epilogue block) failed (%d): ptr=%p elem=%d dims=[%llu,%llu,%llu] strides=[%llu,%llu]", (int)r, ptr, elem_bytes,
              (unsigned long long)gdim[0], (unsigned long long)gdim[1], (unsigned long long)gdim[2], (unsigned long long)gstride[0],
              (unsigned long long)gstride[1]);
    return -3;
  }
  if (g_bm_cache.size() > 8192) g_bm_cache.clear();
  g_bm_cache[key] = tm;
  *out = tm;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// GEMM front end: C[M,N] = A[M,K] * B[N,K]^T through `epi`, on the engine the activation type selects
// ------------------------------------------------------------------------------------------------
enum GemmMode { G_FWD = 0 /* A K-major, B K-major */, G_DGRAD = 1 /* A K-major, B MN-major */, G_WGRAD = 2 /* both MN-major */ };

template <typename T> struct Engine;

template <> struct Engine<float> {
  template <int MODE, class Epi>
  static int gemm(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int N, int64_t K, int splits, bool vec_ok,
                  const Epi& epi, cudaStream_t st) {
    constexpr bool a_mn = (MODE == G_WGRAD), b_mn = (MODE != G_FWD);
    SgemmOperand a{A, a_mn ? 1 : lda, a_mn ? lda : 1};
    SgemmOperand b{B, b_mn ? 1 : ldb, b_mn ? ldb : 1};
    return sgemm_launch(a, b, M, N, K, splits, vec_ok, epi, st);
  }
  static int wgrad_splits(int64_t M, int64_t N, int64_t K) {
    const int64_t tiles = ceil_div64(M, SG_BM) * ceil_div64(N, SG_BN);
    int64_t s = ceil_div64(2 * PSVAE_NUM_SMS, tiles);
    if (s < ceil_div64(K, 2048)) s = ceil_div64(K, 2048);  // parity engine: short fp32 accumulation chains (<= 2048 rows per partial)
    const int64_t max_s = K / 128 > 1 ? K / 128 : 1;      // at least 128 rows per split
    if (s > max_s) s = max_s;
    if (s > g_opt.wgrad_split_cap) s = g_opt.wgrad_split_cap;
    if (s < 1) s = 1;
    const int64_t chunk = align_up64(ceil_div64(K, s), SG_BK);
    return (int)ceil_div64(K, chunk);
  }
};

template <> struct Engine<bf16> {
  template <int MODE, class Epi>
  static int gemm(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int64_t M, int N, int64_t K, int splits, bool /*vec_ok*/,
                  const Epi& epi, cudaStream_t st) {
    constexpr bool a_mn = (MODE == G_WGRAD), b_mn = (MODE != G_FWD);
    TcOperand a{A, M, lda, a_mn};
    TcOperand b{B, (int64_t)N, ldb, b_mn};
    return gemm_tc_launch<a_mn, b_mn, Epi>(a, b, M, N, K, splits, epi, st, (int)g_opt.tc_force_bn);
  }
  // block-diagonal pair (the two encoders): A [M][groups * Kg], C [M][groups * Ng], weights stacked; see TcShape::groups
  template <int MODE, class Epi>
  static int gemm_grouped(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int64_t M, int groups, int Ng, int Kg, int64_t out_group_stride,
                          const Epi& epi, cudaStream_t st) {
    static_assert(MODE != G_WGRAD, "grouped launches: forward and dgrad forms");
    constexpr bool b_mn = (MODE != G_FWD);
    TcOperand a{A, M, lda, false};
    TcOperand b{B, b_mn ? (int64_t)Ng : (int64_t)groups * Ng, ldb, b_mn};
    TcGroup g;
    g.groups = groups; g.grp_n = Ng; g.grp_k = Kg; g.out_group_stride = out_group_stride;
    return gemm_tc_launch<false, b_mn, Epi>(a, b, M, groups * Ng, Kg, 1, epi, st, (int)g_opt.tc_force_bn, g);
  }
  static bool grouped_ok(int Ng, int Kg) {
    const int bn = g_opt.tc_force_bn ? (int)g_opt.tc_force_bn : tc_pick_bn(Ng);
    return g_opt.tc_grouped && Ng % bn == 0 && Kg % TC_BK == 0;
  }
  static int wgrad_splits(int64_t M, int64_t N, int64_t K) {
    const int bn = g_opt.tc_force_bn ? (int)g_opt.tc_force_bn : tc_pick_bn((int)N);
    const int cg = tc_use_pair(M, (int)N, (int)g_opt.tc_force_bn) ? 2 : 1;
    const int64_t tiles = ceil_div64(M, TC_BM * cg) * ceil_div64(N, bn);
    const int64_t kb = ceil_div64(K, TC_BK);
    int64_t s = (PSVAE_NUM_SMS / cg) / tiles;
    if (s > kb) s = kb;
    if (s > g_opt.wgrad_split_cap) s = g_opt.wgrad_split_cap;
    if (s < 1) s = 1;
    const int64_t per = ceil_div64(kb, s);
    return (int)ceil_div64(kb, per);          // no empty split
  }
};

// ------------------------------------------------------------------------------------------------
// model shape helpers
// ------------------------------------------------------------------------------------------------
struct Net {
  const psvae_model_desc* d;
  int D, L, H, nh;             // nh hidden layers => nh + 1 Linear layers per MLP
  explicit Net(const psvae_model_desc* desc) : d(desc), D(desc->input_dim), L(desc->latent_dim), H(desc->hidden_dim), nh(desc->num_hidden) {}
  int enc_in(int j) const { return j == 0 ? D : H; }
  int enc_out(int j) const { return j == nh ? L : H; }
  int dec_in(int j) const { return j == 0 ? L : H; }
  int dec_out(int j) const { return j == nh ? D : H; }
  bool has_clf() const { return d->clf_num_heads > 0; }
  int clf_feat() const { return d->clf_num_trunk > 0 ? d->clf_hidden : L; }
  int clf_trunk_in(int t) const { return t == 0 ? L : d->clf_hidden; }
};

static int check_desc(const psvae_model_desc* d, int precision) {
  if (!d) { set_error("desc is NULL"); return -1; }
  if (d->input_dim < 4 || d->input_dim % 4) { set_error("input_dim=%d must be a positive multiple of 4", d->input_dim); return -2; }
  if (d->latent_dim < 4 || d->latent_dim % 4 || d->latent_dim > 256) { set_error("latent_dim=%d must be a multiple of 4 in [4,256]", d->latent_dim); return -2; }
  if (d->hidden_dim < 4 || d->hidden_dim % 4) { set_error("hidden_dim=%d must be a positive multiple of 4", d->hidden_dim); return -2; }
  if (d->num_hidden < 1 || d->num_hidden + 1 > PSVAE_MAX_LAYERS) { set_error("num_hidden=%d out of range [1,%d]", d->num_hidden, PSVAE_MAX_LAYERS - 1); return -2; }
  if (d->clf_num_heads < 0 || d->clf_num_heads > PSVAE_MAX_CLF_HEADS) { set_error("clf_num_heads=%d out of range", d->clf_num_heads); return -2; }
  if (d->clf_num_trunk < 0 || d->clf_num_trunk > PSVAE_MAX_CLF_TRUNK) { set_error("clf_num_trunk=%d out of range", d->clf_num_trunk); return -2; }
  if (d->clf_num_heads > 0) {
    if (d->clf_num_trunk > 0 && (d->clf_hidden < 1 || d->clf_hidden > 1024)) { set_error("clf_hidden=%d out of range [1,1024]", d->clf_hidden); return -2; }
    if (d->clf_activation < 0 || d->clf_activation > 3) { set_error("clf_activation=%d unknown", d->clf_activation); return -2; }
    for (int h = 0; h < d->clf_num_heads; ++h) {
      if (d->clf_head_classes[h] < 2) {
        // the reference's 1-logit "binary" branch is degenerate (log_softmax of one logit == 0; SURVEY F11)
        set_error("classifier head %d has %d classes; at least 2 are required", h, d->clf_head_classes[h]);
        return -2;
      }
      if (d->clf_head_classes[h] > LG_MAXC) { set_error("classifier head %d has %d classes; at most %d are supported", h, d->clf_head_classes[h], LG_MAXC); return -2; }
    }
  }
  if (precision == PSVAE_BF16) {
    if (d->input_dim % 8 || d->latent_dim % 8 || d->hidden_dim % 64) {
      set_error("PSVAE_BF16 needs input_dim %% 8 == 0, latent_dim %% 8 == 0, hidden_dim %% 64 == 0 (got %d, %d, %d)", d->input_dim, d->latent_dim, d->hidden_dim);
      return -2;
    }
  } else if (precision != PSVAE_FP32) {
    set_error("unknown precision %d", precision);
    return -2;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// workspace carving (the caller owns the memory; the same function sizes and carves)
// ------------------------------------------------------------------------------------------------
struct Bump {
  char* base;
  int64_t used = 0;
  explicit Bump(void* b) : base(static_cast<char*>(b)) {}
  template <typename T> T* take(int64_t n) {
    const int64_t off = used;
    used = align_up64(used + n * (int64_t)sizeof(T), 256);
    return base ? reinterpret_cast<T*>(base + off) : nullptr;
  }
};

template <typename TAct> struct StepBufs {
  TAct* xa = nullptr;
  TAct* he[PSVAE_MAX_LAYERS] = {};
  float *mu = nullptr, *ls = nullptr;
  TAct* z = nullptr;
  TAct* hs = nullptr;             // sigma * eps / 2 (training): what the backward pass needs of the reparameterisation
  TAct* hd[PSVAE_MAX_LAYERS] = {};
  float* u = nullptr;
  TAct* dxh = nullptr;
  TAct* gd[2] = {};
  float *dz = nullptr, *dmu_clf = nullptr;
  TAct *dmu = nullptr, *dls = nullptr;
  TAct* ge[2] = {};
  float* clf_act[PSVAE_MAX_CLF_TRUNK] = {};
  float* logits[PSVAE_MAX_CLF_HEADS] = {};
  float* clf_g[2] = {};
  float *wpart = nullptr, *cpart = nullptr;
  float *clf_part = nullptr, *clf_sums = nullptr;
  float* clf_grows = nullptr;      // option clf_grad_in_bwd: d loss / d logits [rows][CLF_MAXC]
  uint32_t* mhe[PSVAE_MAX_LAYERS] = {};   // ReLU bit masks of the hidden activations (tcgen05 training): [features/32][rows]
  uint32_t* mhd[PSVAE_MAX_LAYERS] = {};     // fused classifier: per-block partials, summed nll/acc
  float *sse_part = nullptr, *kl_part = nullptr, *nll_part[PSVAE_MAX_CLF_HEADS] = {}, *acc_part[PSVAE_MAX_CLF_HEADS] = {};
  int64_t n_sse = 0, n_kl = 0, n_ce = 0;
  // option tc_merged_wgrad: the wgrad problems collected during the backward pass, launched together (flushed earlier only before a
  // ping-pong gradient buffer they read is overwritten: more than two hidden layers)
  TcWgradProblem pending[TC_MAX_PROBLEMS];
  int n_pending = 0;
  bool merge_wgrads = false;
};

template <typename TAct>
static int flush_wgrads(StepBufs<TAct>& w, int64_t rows, cudaStream_t st) {
  if (w.n_pending == 0) return 0;
  const int n = w.n_pending;
  w.n_pending = 0;
  // option wgrad_order: 1 = newest gradient first (the tensors the backward pass wrote last are the ones still in L2), 2 = and each problem's
  // batch ranges from the end
  if (g_opt.wgrad_order >= 1)
    for (int i = 0; i < n / 2; ++i) std::swap(w.pending[i], w.pending[n - 1 - i]);
  return gemm_tc_launch_multi_wgrad(w.pending, n, rows, st, g_opt.wgrad_order >= 2 ? 1 : 0);
}

// the fused classifier kernel covers the common shape: heads directly on mu (no trunk), L = 16/32/64/128, <= 8 classes in total
static bool clf_fused_ok(const psvae_model_desc* d) {
  if (d->clf_num_heads <= 0 || d->clf_num_trunk != 0) return false;
  if (d->latent_dim != 16 && d->latent_dim != 32 && d->latent_dim != 64 && d->latent_dim != 128) return false;   // kernel instantiations
  int total = 0;
  for (int h = 0; h < d->clf_num_heads; ++h) total += d->clf_head_classes[h];
  return total <= CLF_MAXC && total * d->latent_dim <= CLF_ACCW * CLF_TILE;
}
static int clf_fused_blocks(int64_t rows) {
  int64_t b = ceil_div64(rows, CLF_TILE);
  if (b > 4 * PSVAE_NUM_SMS) b = 4 * PSVAE_NUM_SMS;
  return b < 1 ? 1 : (int)b;
}
// the 8-columns-per-thread latent backward (latent_bwd_clf8_kernel): L a multiple of 8 with L / 8 dividing 256, at most 4 classes in total
static bool latent8_ok(int L, int total_classes) { return L % 8 == 0 && 256 % (L / 8) == 0 && L <= 256 && total_classes >= 1 && total_classes <= 4; }
static bool latent_cs_ok(int L) { return L % 4 == 0 && 256 % (L / 4) == 0 && 2 * L <= 256; }
// Does the tcgen05 train step of this model use the fused encoder-head kernel (EpiLatent)?  Decided from the model shape and the options only
// (so that the workspace plan and the step agree): latent 64, hidden a multiple of 64, no classifier or ONE linear head of <= 4 classes.
static bool fused_head_shape_ok(const psvae_model_desc* d) {
  if (!g_opt.fused_head || g_opt.deterministic) return false;
  if (d->latent_dim != TC_LAT_L || d->hidden_dim % TC_BK != 0) return false;
  if (d->clf_num_heads > 0 && !(clf_fused_ok(d) && d->clf_num_heads == 1 && d->clf_head_classes[0] <= 4 && latent_cs_ok(d->latent_dim))) return false;
  return true;
}
// the [rows][CLF_MAXC] d loss / d logits buffer exists when the classifier's backward runs inside the latent backward kernel
static bool clf_rows_wanted(const psvae_model_desc* d) { return clf_fused_ok(d) && (g_opt.clf_grad_in_bwd || fused_head_shape_ok(d)); }

static int64_t sse_slots(int64_t rows, int D) {
  int64_t a = sgemm_red_slots(rows, D);
  int64_t b = ceil_div64(rows * 32, 256);     // recon_rows_kernel: 8 rows per block
  int64_t c = PSVAE_NUM_SMS * 2;              // tcgen05 engine: one per CTA
  return a > b ? (a > c ? a : c) : (b > c ? b : c);
}

template <typename TAct>
static void plan(const psvae_model_desc* d, int64_t rows, int mode, Bump& b, StepBufs<TAct>& w) {
  Net n(d);
  const bool is_bf16 = sizeof(TAct) == 2;
  if (mode == PSVAE_MODE_DECODE) {
    w.z = b.take<TAct>(rows * n.L);
    for (int j = 0; j < n.nh; ++j) w.hd[j] = b.take<TAct>(rows * n.H);
    return;
  }
  const bool train = (mode == PSVAE_MODE_TRAIN);
  const bool clf_train = (mode == PSVAE_MODE_TRAIN_CLASSIFIER);
  if (is_bf16) w.xa = b.take<TAct>(rows * n.D);
  for (int j = 0; j < n.nh; ++j) w.he[j] = b.take<TAct>(rows * 2 * n.H);
  w.mu = b.take<float>(rows * n.L);
  w.ls = b.take<float>(rows * n.L);
  w.z = b.take<TAct>(rows * n.L);
  for (int j = 0; j < n.nh; ++j) w.hd[j] = b.take<TAct>(rows * n.H);
  w.u = b.take<float>(rows * n.D);
  w.n_sse = sse_slots(rows, n.D);
  w.n_kl = ew_grid(rows * n.L / 4);
  w.n_ce = ceil_div64(rows, 256);
  w.sse_part = b.take<float>(w.n_sse);
  w.kl_part = b.take<float>(w.n_kl);
  if (n.has_clf()) {
    if (clf_fused_ok(d)) {
      w.clf_part = b.take<float>((int64_t)clf_fused_blocks(rows) * clf_part_len(n.L));
      w.clf_sums = b.take<float>(8);
    } else {
      for (int t = 0; t < d->clf_num_trunk; ++t) w.clf_act[t] = b.take<float>(rows * d->clf_hidden);
      for (int h = 0; h < d->clf_num_heads; ++h) {
        w.logits[h] = b.take<float>(rows * d->clf_head_classes[h]);
        w.nll_part[h] = b.take<float>(w.n_ce);
        w.acc_part[h] = b.take<float>(w.n_ce);
      }
    }
  }
  if (clf_train && n.has_clf()) {
    // the classifier's backward only.  The fused encoder head (fast mode) stays the forward kernel: it writes sigma eps / 2 next to z
    // through one 3D output map (so it needs that buffer, right after z) and d loss / d logits per row
    if (is_bf16 && fused_head_shape_ok(d)) {
      w.hs = b.take<TAct>(rows * n.L);
      w.clf_grows = b.take<float>(rows * CLF_MAXC);
    }
    if (!clf_fused_ok(d)) {
      int64_t wmax = 0, cmax = d->clf_hidden;
      auto upd = [&](int64_t M, int64_t N) {
        const int64_t s = Engine<float>::wgrad_splits(M, N, rows);
        if (s * M * N > wmax) wmax = s * M * N;
      };
      if (d->clf_num_trunk > 0) for (int i = 0; i < 2; ++i) w.clf_g[i] = b.take<float>(rows * d->clf_hidden);
      for (int t = 0; t < d->clf_num_trunk; ++t) upd(d->clf_hidden, n.clf_trunk_in(t));
      for (int h = 0; h < d->clf_num_heads; ++h) {
        upd(d->clf_head_classes[h], n.clf_feat());
        if (d->clf_head_classes[h] > cmax) cmax = d->clf_head_classes[h];
      }
      w.wpart = b.take<float>(wmax);
      w.cpart = b.take<float>(ceil_div64(rows, g_opt.colsum_rows) * cmax);
    }
    return;
  }
  if (!train) return;
  if (is_bf16) {
    for (int j = 0; j < n.nh; ++j) {
      w.mhe[j] = b.take<uint32_t>((int64_t)(2 * n.H / 32) * rows);
      w.mhd[j] = b.take<uint32_t>((int64_t)(n.H / 32) * rows);
    }
  }
  w.hs = b.take<TAct>(rows * n.L);
  w.dxh = b.take<TAct>(rows * n.D);
  for (int i = 0; i < 2; ++i) w.gd[i] = b.take<TAct>(rows * n.H);
  w.dz = b.take<float>(rows * n.L);
  w.dmu = b.take<TAct>(rows * 2 * n.L);        // [rows][2L]: dmu | dls side by side (one A operand for the grouped encoder-head dgrad)
  w.dls = w.dmu ? w.dmu + n.L : nullptr;
  for (int i = 0; i < 2; ++i) w.ge[i] = b.take<TAct>(rows * 2 * n.H);
  int64_t wmax = 0, cmax = 2 * n.H > n.D ? 2 * n.H : n.D;
  auto upd = [&](int64_t M, int64_t N, bool clf) {
    const int s = clf ? Engine<float>::wgrad_splits(M, N, rows) : Engine<TAct>::wgrad_splits(M, N, rows);
    if (s * M * N > wmax) wmax = s * M * N;
  };
  upd(2 * n.enc_out(0), n.enc_in(0), false);
  for (int j = 1; j <= n.nh; ++j) upd(n.enc_out(j), n.enc_in(j), false);
  for (int j = 0; j <= n.nh; ++j) upd(n.dec_out(j), n.dec_in(j), false);
  if (n.has_clf()) {
    if (clf_rows_wanted(d)) w.clf_grows = b.take<float>(rows * CLF_MAXC);
    w.dmu_clf = b.take<float>(rows * n.L);
    if (!clf_fused_ok(d)) {
      const int gw = d->clf_hidden > n.L ? d->clf_hidden : n.L;
      for (int i = 0; i < 2; ++i) w.clf_g[i] = b.take<float>(rows * gw);
      for (int t = 0; t < d->clf_num_trunk; ++t) upd(d->clf_hidden, n.clf_trunk_in(t), true);
      for (int h = 0; h < d->clf_num_heads; ++h) upd(d->clf_head_classes[h], n.clf_feat(), true);
      if (d->clf_hidden > cmax) cmax = d->clf_hidden;
    }
  }
  w.wpart = b.take<float>(wmax);
  // bias-gradient partials: [row chunks][N] from colsum_kernel, [CTAs][N] from the tcgen05 epilogues, [blocks][2L] from latent_bwd_cs
  int64_t cslots = ceil_div64(rows, g_opt.colsum_rows);
  if (cslots < 4 * 160) cslots = 4 * 160;        // tcgen05 epilogues: one partial row per (CTA, TMEM lane quarter)
  const int64_t lat = (int64_t)PSVAE_NUM_SMS * 8 * 2 * n.L;
  w.cpart = b.take<float>(cslots * cmax > lat ? cslots * cmax : lat);
}

// ------------------------------------------------------------------------------------------------
// small launch helpers
// ------------------------------------------------------------------------------------------------
static int launch_reduce(const float* partials, int64_t n, int S, float* out, cudaStream_t st);
template <typename T>
static int launch_colsum(const T* in, int64_t ld, int64_t rows, int N, float* cpart, float* out, cudaStream_t st) {
  const int64_t rpc = g_opt.colsum_rows;
  const int chunks = (int)ceil_div64(rows, rpc);
  dim3 grid((unsigned)ceil_div64(N, 32), (unsigned)chunks);
  launch_dep(colsum_kernel<T>, dim3(grid), dim3(256), 0, st, in, ld, rows, N, rpc, cpart);
  count_launch();
  PSVAE_LAUNCH_CHECK("colsum_kernel");
  return launch_reduce(cpart, N, chunks, out, st);
}
static int launch_reduce(const float* partials, int64_t n, int S, float* out, cudaStream_t st) {
  if (S >= 32 && n <= 65536) {       // many partial rows, few columns: spread the rows over the block (fixed-order tree)
    launch_dep(reduce_tall_kernel, dim3((unsigned)ceil_div64(n, 32)), dim3(1024), 0, st, partials, (int)n, S, n, out);
    count_launch();
    PSVAE_LAUNCH_CHECK("reduce_tall_kernel");
    return 0;
  }
  launch_dep(reduce_partials_kernel, dim3((unsigned)ceil_div64(n, 256)), dim3(256), 0, st, partials, n, S, n, 1.f, out);
  count_launch();
  PSVAE_LAUNCH_CHECK("reduce_partials_kernel");
  return 0;
}

// dW[M=out][N=in] = dY[B][out]^T * A[B][in]   (+ bias gradient = column sums of dY)
template <typename TAct>
static int wgrad(const TAct* dY, int64_t ldy, const TAct* A, int64_t lda, int64_t rows, int out, int in, float* gW, float* gb,
                 StepBufs<TAct>& w, cudaStream_t st) {
  if (sizeof(TAct) == 2 && w.merge_wgrads) {
    if (w.n_pending == TC_MAX_PROBLEMS) PSVAE_TRY(flush_wgrads(w, rows, st));
    w.pending[w.n_pending++] = TcWgradProblem{dY, ldy, A, lda, gW, (int64_t)in, out, in};
    if (!gb) return 0;
    return launch_colsum<TAct>(dY, ldy, rows, out, w.cpart, gb, st);
  }
  const int splits = Engine<TAct>::wgrad_splits(out, in, rows);
  if (sizeof(TAct) == 2 && !g_opt.deterministic) {
    // fast mode: every split-K tile adds its block into the (zeroed) gradient with a TMA reduce-add -- no partial buffers, no second pass
    EpiStore e{gW, in, 0, 1.f, 0.f, nullptr, 1};
    PSVAE_TRY((Engine<TAct>::template gemm<G_WGRAD>(dY, ldy, A, lda, out, in, rows, splits, in % 4 == 0, e, st)));
  } else if (splits == 1) {
    EpiStore e{gW, in, 0, 1.f, 0.f, nullptr, 0};
    PSVAE_TRY((Engine<TAct>::template gemm<G_WGRAD>(dY, ldy, A, lda, out, in, rows, 1, in % 4 == 0, e, st)));
  } else {
    EpiStore e{w.wpart, in, (int64_t)out * in, 1.f, 0.f, nullptr, 0};
    PSVAE_TRY((Engine<TAct>::template gemm<G_WGRAD>(dY, ldy, A, lda, out, in, rows, splits, in % 4 == 0, e, st)));
    PSVAE_TRY(launch_reduce(w.wpart, (int64_t)out * in, splits, gW, st));
  }
  if (!gb) return 0;        // the kernel that produced dY already emitted its column sums
  return launch_colsum<TAct>(dY, ldy, rows, out, w.cpart, gb, st);
}

// dgrad through a hidden Linear: out[B][in] = (dY[B][out] W[out][in]) .* relu'(act).  In tcgen05 mode the epilogue also emits the
// column sums of `out` (= bias gradient of the layer below) into `bias_grad`; *bias_done tells the caller whether it did.
template <typename TAct>
static int dgrad_hidden(const TAct* dY, int64_t ldy, const TAct* W, int out_dim, int in_dim, const TAct* act, int64_t lda, const uint32_t* mask,
                        TAct* out, int64_t ldo, int64_t rows, float* bias_grad, StepBufs<TAct>& w, bool* bias_done, cudaStream_t st) {
  *bias_done = false;
  if constexpr (sizeof(TAct) == 2) {
    if (bias_grad && tc_colsum_ok(in_dim)) {
      const bool atomic = !g_opt.deterministic;
      EpiActGrad<TAct, TAct, ACT_RELU, true> e{act, lda, mask, rows, out, ldo, 0.f, nullptr, atomic ? bias_grad : w.cpart, atomic ? 1 : 0};
      PSVAE_TRY((Engine<TAct>::template gemm<G_DGRAD>(dY, ldy, W, in_dim, rows, in_dim, out_dim, 1, true, e, st)));
      if (!atomic) {
        const int64_t ctas = tc_ctas(rows, in_dim, 1, (int)g_opt.tc_force_bn);
        PSVAE_TRY(launch_reduce(w.cpart, in_dim, (int)ctas * 4, bias_grad, st));
      }
      *bias_done = true;
      return 0;
    }
  }
  EpiActGrad<TAct, TAct, ACT_RELU, false> e{act, lda, mask, rows, out, ldo, 0.f, nullptr, nullptr, 0};
  return Engine<TAct>::template gemm<G_DGRAD>(dY, ldy, W, in_dim, rows, in_dim, out_dim, 1, true, e, st);
}
// classifier wgrad: always fp32 on the CUDA cores
template <typename TAct>
static int wgrad_clf(const float* dY, int64_t ldy, const float* A, int64_t lda, int64_t rows, int out, int in, float* gW, float* gb,
                     StepBufs<TAct>& w, cudaStream_t st) {
  const int splits = Engine<float>::wgrad_splits(out, in, rows);
  const bool vec = (in % 4 == 0);
  if (splits == 1) {
    EpiStore e{gW, in, 0, 1.f, 0.f, nullptr, 0};
    PSVAE_TRY((Engine<float>::gemm<G_WGRAD>(dY, ldy, A, lda, out, in, rows, 1, vec, e, st)));
  } else {
    EpiStore e{w.wpart, in, (int64_t)out * in, 1.f, 0.f, nullptr, 0};
    PSVAE_TRY((Engine<float>::gemm<G_WGRAD>(dY, ldy, A, lda, out, in, rows, splits, vec, e, st)));
    PSVAE_TRY(launch_reduce(w.wpart, (int64_t)out * in, splits, gW, st));
  }
  return launch_colsum<float>(dY, ldy, rows, out, w.cpart, gb, st);
}

template <int ACT>
static int clf_linear_act(const float* a, int64_t lda, const float* W, const float* b, float* out, int64_t rows, int N, int K, cudaStream_t st) {
  EpiBiasAct<float, ACT> e{b, out, N, nullptr};
  return Engine<float>::gemm<G_FWD>(a, lda, W, K, rows, N, K, 1, N % 4 == 0, e, st);
}
static int clf_linear(int act, const float* a, int64_t lda, const float* W, const float* b, float* out, int64_t rows, int N, int K, cudaStream_t st) {
  switch (act) {
    case ACT_NONE: return clf_linear_act<ACT_NONE>(a, lda, W, b, out, rows, N, K, st);
    case ACT_RELU: return clf_linear_act<ACT_RELU>(a, lda, W, b, out, rows, N, K, st);
    case ACT_TANH: return clf_linear_act<ACT_TANH>(a, lda, W, b, out, rows, N, K, st);
    case ACT_SIGMOID: return clf_linear_act<ACT_SIGMOID>(a, lda, W, b, out, rows, N, K, st);
    case ACT_LEAKY: return clf_linear_act<ACT_LEAKY>(a, lda, W, b, out, rows, N, K, st);
  }
  set_error("unknown activation %d", act);
  return -2;
}
// out[B][in] = (dY[B][out] * W[out][in]) .* act'(A[B][in]) + beta * out
template <int ACT>
static int clf_dgrad_act(const float* dY, int out_dim, const float* W, int in_dim, const float* A, float* out, float beta, int64_t rows, cudaStream_t st) {
  EpiActGrad<float, float, ACT> e{A, in_dim, nullptr, 0, out, in_dim, beta, nullptr, nullptr, 0};
  return Engine<float>::gemm<G_DGRAD>(dY, out_dim, W, in_dim, rows, in_dim, out_dim, 1, in_dim % 4 == 0, e, st);
}
static int clf_dgrad(int act, const float* dY, int out_dim, const float* W, int in_dim, const float* A, float* out, float beta, int64_t rows, cudaStream_t st) {
  if (!A) {
    EpiStore e{out, in_dim, 0, 1.f, beta, nullptr, 0};
    return Engine<float>::gemm<G_DGRAD>(dY, out_dim, W, in_dim, rows, in_dim, out_dim, 1, in_dim % 4 == 0, e, st);
  }
  switch (act) {
    case ACT_RELU: return clf_dgrad_act<ACT_RELU>(dY, out_dim, W, in_dim, A, out, beta, rows, st);
    case ACT_TANH: return clf_dgrad_act<ACT_TANH>(dY, out_dim, W, in_dim, A, out, beta, rows, st);
    case ACT_SIGMOID: return clf_dgrad_act<ACT_SIGMOID>(dY, out_dim, W, in_dim, A, out, beta, rows, st);
    case ACT_LEAKY: return clf_dgrad_act<ACT_LEAKY>(dY, out_dim, W, in_dim, A, out, beta, rows, st);
  }
  set_error("unknown activation %d", act);
  return -2;
}

// ------------------------------------------------------------------------------------------------
// consistency classifier (frozen EmbeddingClassifier, embedding_classifier.py:29-62): fp32 on the CUDA cores in both precisions
// ------------------------------------------------------------------------------------------------
struct ConsBufs {
  float* xh = nullptr;            // normalised x_hat when the caller did not ask for it
  float *a1 = nullptr, *a2 = nullptr, *logits = nullptr;
  float *g2 = nullptr, *g1 = nullptr, *gx = nullptr;
  float *nll_part = nullptr, *acc_part = nullptr;
  int64_t n_ce = 0;
};
static int check_cons(const psvae_consistency_desc* c) {
  if (!c) { set_error("consistency desc is NULL"); return -1; }
  if (c->input_dim < 4 || c->input_dim % 4) { set_error("consistency input_dim=%d must be a positive multiple of 4", c->input_dim); return -2; }
  if (c->hidden_dim < 4 || c->hidden_dim % 4) { set_error("consistency hidden_dim=%d must be a positive multiple of 4", c->hidden_dim); return -2; }
  if (c->num_classes < 2) { set_error("consistency num_classes=%d must be at least 2", c->num_classes); return -2; }
  return 0;
}
static void plan_cons(const psvae_consistency_desc* c, int64_t rows, bool train, Bump& b, ConsBufs& w) {
  w.xh = b.take<float>(rows * c->input_dim);
  w.a1 = b.take<float>(rows * c->hidden_dim);
  w.a2 = b.take<float>(rows * c->hidden_dim);
  w.logits = b.take<float>(rows * c->num_classes);
  w.n_ce = ceil_div64(rows, 256);
  w.nll_part = b.take<float>(w.n_ce);
  w.acc_part = b.take<float>(w.n_ce);
  if (!train) return;
  w.g2 = b.take<float>(rows * c->hidden_dim);
  w.g1 = b.take<float>(rows * c->hidden_dim);
  w.gx = b.take<float>(rows * c->input_dim);
}
// logits = fc3(relu(fc2(relu(fc1(xh)))))
static int cons_forward(const psvae_consistency_desc* c, const float* cp, const float* xh, int64_t rows, ConsBufs& w, float* logits, cudaStream_t st) {
  PSVAE_TRY(clf_linear(ACT_RELU, xh, c->input_dim, cp + c->w[0], cp + c->b[0], w.a1, rows, c->hidden_dim, c->input_dim, st));
  PSVAE_TRY(clf_linear(ACT_RELU, w.a1, c->hidden_dim, cp + c->w[1], cp + c->b[1], w.a2, rows, c->hidden_dim, c->hidden_dim, st));
  return clf_linear(ACT_NONE, w.a2, c->hidden_dim, cp + c->w[2], cp + c->b[2], logits, rows, c->num_classes, c->hidden_dim, st);
}
// gx = d loss / d x_hat given dlogits (in w.logits); no parameter gradients (the classifier is frozen)
static int cons_input_grad(const psvae_consistency_desc* c, const float* cp, int64_t rows, ConsBufs& w, cudaStream_t st) {
  PSVAE_TRY(clf_dgrad(ACT_RELU, w.logits, c->num_classes, cp + c->w[2], c->hidden_dim, w.a2, w.g2, 0.f, rows, st));
  PSVAE_TRY(clf_dgrad(ACT_RELU, w.g2, c->hidden_dim, cp + c->w[1], c->hidden_dim, w.a1, w.g1, 0.f, rows, st));
  return clf_dgrad(ACT_NONE, w.g1, c->hidden_dim, cp + c->w[0], c->input_dim, nullptr, w.gx, 0.f, rows, st);
}

// ------------------------------------------------------------------------------------------------
// the step: forward (+ losses) (+ backward)
// ------------------------------------------------------------------------------------------------
struct StepArgs {
  const psvae_model_desc* d;
  const float* params;
  const bf16* shadow;
  float* grads;
  const float* x;            // fp32 input [rows][D] ...
  const int64_t* y;
  const float* eps;
  uint64_t seed, offset;
  int64_t row0, rows;
  float kl_w, clf_w;
  int use_cos, want_loss, want_grads;
  float *x_hat, *mu, *ls, *losses;
  void* ws;
  int64_t ws_bytes;
  cudaStream_t st;
  // consistency classifier on x_hat (lightning.py:44-52, 100-108); cons == nullptr: none
  const psvae_consistency_desc* cons = nullptr;
  const float* cons_params = nullptr;
  const int64_t* cons_y = nullptr;
  float cons_w = 0.f;
  // backward of VAEModel.forward for a caller's own loss (want_loss = 0, want_grads = 1): d loss / d (x_hat, mu, log_sigma), each optional
  int ext = 0;
  const float* ext_gx = nullptr;
  const float* ext_gmu = nullptr;
  const float* ext_gls = nullptr;
  // ... or the same batch already in bf16 (PSVAE_X_BF16; tensor-core mode only): the operand of the first GEMM as it is, no cast pass, and the
  // reconstruction target of the MSE epilogue (the data ARE these bf16 values: a bf16 embedding store, data.py)
  const bf16* x16 = nullptr;
  // device step counters (psvae_train_fwd_bwd_dc): the Philox offset of the eps draw is read from here instead of `offset`
  const uint64_t* offset_dev = nullptr;
  // PSVAE_GRAD_CLASSIFIER (frozen VAE): the full forward and losses, then only the latent classifier's gradients, into its span of grads
  int grad_scope = PSVAE_GRAD_ALL;
};

template <typename TAct> static const TAct* weights_of(const StepArgs& a);
template <> const float* weights_of<float>(const StepArgs& a) { return a.params; }
template <> const bf16* weights_of<bf16>(const StepArgs& a) { return a.shadow; }

// decoder chain z -> pre-normalisation output; the last layer goes through `last_epi`
template <typename TAct, class LastEpi>
static int decoder_forward(const Net& n, const TAct* Wt, const float* params, const TAct* z, TAct* const* hd, int64_t rows, const LastEpi& last_epi,
                           cudaStream_t st, uint32_t* const* mhd = nullptr) {
  const TAct* a = z;
  for (int j = 0; j < n.nh; ++j) {
    EpiBiasAct<TAct, ACT_RELU> e{params + n.d->dec_b[j], hd[j], n.H, nullptr, mhd ? mhd[j] : nullptr, rows};
    PSVAE_TRY((Engine<TAct>::template gemm<G_FWD>(a, n.dec_in(j), Wt + n.d->dec_w[j], n.dec_in(j), rows, n.H, n.dec_in(j), 1, true, e, st)));
    a = hd[j];
  }
  return Engine<TAct>::template gemm<G_FWD>(a, n.H, Wt + n.d->dec_w[n.nh], n.H, rows, n.D, n.H, 1, n.D % 4 == 0, last_epi, st);
}

// clf_fused_kernel<REPARAM> with its dynamic shared memory; GROWS: option clf_grad_in_bwd, DEV_OFF: device step counters
template <int LL, typename TAct, bool GROWS, bool DEV_OFF>
static int launch_clf_fused(int blocks, size_t smem, cudaStream_t st, const float* P, const float* mu, const int64_t* y, int64_t B, const ClfFusedArgs& ca,
                            float* dmu_out, float* part, const ReparamArgs& rp) {
  auto kern = clf_fused_kernel<LL, TAct, true, GROWS, DEV_OFF>;
  PSVAE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_dep(kern, dim3(blocks), dim3(CLF_TILE), smem, st, P, mu, y, B, ca, dmu_out, part, rp);
  return 0;
}

template <typename TAct>
static int run_step(const StepArgs& a) {
  PSVAE_TRY(tc_device_check());
  const psvae_model_desc* d = a.d;
  Net n(d);
  const int64_t B = a.rows;
  cudaStream_t st = a.st;
  if (B <= 0) { set_error("rows=%lld must be positive", (long long)B); return -2; }
  if (!a.params || !(a.x || a.x16)) { set_error("params and x must not be NULL"); return -1; }
  if (a.x16 && sizeof(TAct) != 2) { set_error("a bf16 input batch needs precision PSVAE_BF16 (the fp32 parity engine takes fp32 x)"); return -2; }
  if (a.x16 && a.want_loss && (d->normalize_decoder || a.use_cos || a.cons)) {
    set_error("a bf16 input batch is supported by the fused MSE tail only (no normalize_decoder / use_cos_loss / consistency classifier): pass fp32 x");
    return -2;
  }
  if (sizeof(TAct) == 2 && !a.shadow) { set_error("PSVAE_BF16 needs the bf16 shadow copy of the parameters (psvae_refresh_shadow)"); return -1; }
  if (a.want_grads && !a.grads) { set_error("grads must not be NULL when compute_grads != 0"); return -1; }
  if (a.want_loss && !a.losses) { set_error("losses must not be NULL"); return -1; }
  if (a.want_loss && n.has_clf() && !a.y) { set_error("y must not be NULL when the model has a classifier"); return -1; }
  // classifier-only scope: the forward half behaves as a forward with losses for everything the VAE backward would read (no ReLU masks, no
  // sigma eps / 2, no d loss / d x_hat); `vae_grads` is what `want_grads` means for the VAE
  const bool clf_only = a.want_grads && a.grad_scope == PSVAE_GRAD_CLASSIFIER;
  if (clf_only && (!n.has_clf() || !a.want_loss || a.ext)) { set_error("the classifier gradient scope needs a model with a latent classifier"); return -2; }
  const bool vae_grads = a.want_grads && !clf_only;
  const int mode = clf_only ? PSVAE_MODE_TRAIN_CLASSIFIER : a.want_grads ? PSVAE_MODE_TRAIN : PSVAE_MODE_FORWARD;
  const bool cons_on = a.cons != nullptr && a.want_loss;
  if (cons_on) {
    PSVAE_TRY(check_cons(a.cons));
    if (a.cons->input_dim != n.D) { set_error("consistency classifier input_dim=%d, the VAE's is %d", a.cons->input_dim, n.D); return -2; }
    if (!a.cons_params || !a.cons_y) { set_error("cons_params and cons_y must not be NULL"); return -1; }
  }
  StepBufs<TAct> w;
  ConsBufs cw;
  {
    Bump sz(nullptr);
    StepBufs<TAct> tmp;
    ConsBufs ctmp;
    plan<TAct>(d, B, mode, sz, tmp);
    if (cons_on) plan_cons(a.cons, B, vae_grads, sz, ctmp);
    if (sz.used > a.ws_bytes || !a.ws) {
      set_error("workspace too small: need %lld bytes, got %lld", (long long)sz.used, (long long)a.ws_bytes);
      return -2;
    }
    Bump b(a.ws);
    plan<TAct>(d, B, mode, b, w);
    if (cons_on) plan_cons(a.cons, B, vae_grads, b, cw);
  }
  const TAct* Wt = weights_of<TAct>(a);
  const float* P = a.params;
  // gradients are accumulated into (TMA reduce-add / atomics in fast tcgen05 mode) or written into a zeroed buffer; padding reads as zero
  // (tcgen05 mode: the operand cast of x below clears the buffer in the same pass -- total_numel is a multiple of 64 and the buffer 16-byte aligned)
  const bool zero_in_cast = sizeof(TAct) == 2 && vae_grads && (reinterpret_cast<uintptr_t>(a.grads) & 15) == 0;
  if (vae_grads && !zero_in_cast) PSVAE_CUDA(cudaMemsetAsync(a.grads, 0, (size_t)d->total_numel * sizeof(float), st));
  // classifier scope: its span of the buffer only, [vae_numel, total_numel) -- every other element keeps its value
  if (clf_only) PSVAE_CUDA(cudaMemsetAsync(a.grads + d->vae_numel, 0, (size_t)(d->total_numel - d->vae_numel) * sizeof(float), st));
  // option fused_head (training, fast mode): encoder heads + reparameterisation + KL + classifier forward in one kernel.  Its 3D output maps
  // step from mu to log_sigma (and from z to sigma eps / 2) by one stride, so it writes the workspace buffers; a caller's mu / log_sigma get a copy.
  bool fused_head = false;
  if constexpr (sizeof(TAct) == 2)
    fused_head = fused_head_shape_ok(d) && a.want_loss && a.want_grads && !a.ext && (!n.has_clf() || w.clf_grows != nullptr) && w.hs > w.z && w.ls > w.mu;
  float* mu = (a.mu && !fused_head) ? a.mu : w.mu;
  float* ls = (a.ls && !fused_head) ? a.ls : w.ls;
  const int64_t first_elem = a.row0 * n.L;

  // ---- encoders (model.py:54-55).  Layer 0 of both encoders is one [2H, D] GEMM.
  const TAct* xa;
  if constexpr (sizeof(TAct) == 2) {
    if (a.x16) {
      xa = a.x16;
      if (zero_in_cast) {      // no cast pass: the same kernel only clears the gradient buffer (5 MB, L2-resident)
        launch_dep(cast_bf16_kernel, dim3(ew_grid(d->total_numel / 4)), dim3(256), 0, st, (const float*)nullptr, (bf16*)nullptr, (int64_t)0, a.grads, d->total_numel);
        count_launch();
        PSVAE_LAUNCH_CHECK("cast_bf16_kernel");
      }
    } else {
      launch_dep(cast_bf16_kernel, dim3(ew_grid(B * n.D / 8)), dim3(256), 0, st, a.x, w.xa, B * n.D, zero_in_cast ? a.grads : (float*)nullptr,
                 zero_in_cast ? d->total_numel : (int64_t)0);
      count_launch();
      PSVAE_LAUNCH_CHECK("cast_bf16_kernel");
      xa = w.xa;
    }
  } else {
    xa = a.x;
  }
  {
    EpiBiasAct<TAct, ACT_RELU> e{P + d->enc_b[0], w.he[0], 2 * n.H, nullptr, a.want_grads ? w.mhe[0] : nullptr, B};
    PSVAE_TRY((Engine<TAct>::template gemm<G_FWD>(xa, n.D, Wt + d->enc_w[0], n.D, B, 2 * n.H, n.D, 1, true, e, st)));
  }
  // Layers 1..n of the two encoders are block-diagonal: in tcgen05 mode both encoders' layer j is ONE grouped launch (group = encoder:
  // its own k range of the shared [B, 2H] activation buffer, its own rows of the stacked weights, its own column range of the output).
  bool grouped_hidden = false, grouped_head = false;
  if constexpr (sizeof(TAct) == 2) {
    grouped_hidden = Engine<TAct>::grouped_ok(n.H, n.H);
    // mu / log_sigma are two buffers: the output map's third coordinate steps from one to the other (16-byte multiple, forward only)
    grouped_head = Engine<TAct>::grouped_ok(n.L, n.H) && ls > mu && ((ls - mu) % 4) == 0;
  }
  for (int j = 1; j < n.nh; ++j) {
    if constexpr (sizeof(TAct) == 2) {
      if (grouped_hidden) {
        EpiBiasAct<TAct, ACT_RELU> e{P + d->enc_b[j], w.he[j], 2 * n.H, nullptr, (a.want_grads && w.mhe[j]) ? w.mhe[j] : nullptr, B};
        PSVAE_TRY((Engine<TAct>::template gemm_grouped<G_FWD>(w.he[j - 1], 2 * n.H, Wt + d->enc_w[j], n.H, B, 2, n.H, n.H, 0, e, st)));
        continue;
      }
    }
    for (int s = 0; s < 2; ++s) {      // s = 0: encoder_mu, 1: encoder_sigma
      EpiBiasAct<TAct, ACT_RELU> e{P + d->enc_b[j] + s * n.H, w.he[j] + s * n.H, 2 * n.H, nullptr,
                                   (a.want_grads && w.mhe[j]) ? w.mhe[j] + (int64_t)s * (n.H / 32) * B : nullptr, B};
      PSVAE_TRY((Engine<TAct>::template gemm<G_FWD>(w.he[j - 1] + s * n.H, 2 * n.H, Wt + d->enc_w[j] + (int64_t)s * n.H * n.H, n.H, B, n.H, n.H, 1, true, e, st)));
    }
  }
  bool head_done = false;
  // option fused_head: encoder heads + reparameterisation + KL + classifier forward in one kernel (training, fast mode)
  int fused_ctas = 0;
  if constexpr (sizeof(TAct) == 2) {
    if (fused_head) {
      auto launch = [&](auto& e) -> int {
        memset(&e, 0, sizeof(e));
        e.out = mu; e.ldo = n.L;
        e.bias = P + d->enc_b[n.nh];
        e.z = w.z;
        e.eps = a.eps; e.seed = a.seed; e.offset = a.offset; e.offset_dev = a.offset_dev; e.first_quad = first_elem >> 2;
        e.L = n.L;
        e.nc = n.has_clf() ? d->clf_head_classes[0] : 0;
        e.clf_w = n.has_clf() ? P + d->clf_head_w[0] : nullptr;
        e.clf_b = n.has_clf() ? P + d->clf_head_b[0] : nullptr;
        e.y = a.y;
        e.gscale = a.clf_w / (float)B;
        e.g_rows = n.has_clf() ? w.clf_grows : nullptr;
        e.kl_part = w.kl_part;
        e.nll_part = n.has_clf() ? w.clf_part : nullptr;
        e.acc_part = n.has_clf() ? w.clf_part + PSVAE_NUM_SMS : nullptr;
        return gemm_tc_launch_latent(w.he[n.nh - 1], 2 * n.H, Wt + d->enc_w[n.nh], n.H, B, e, mu, ls, w.z, w.hs, st, &fused_ctas);
      };
      if (a.offset_dev) {
        EpiLatent<TAct, true> e;
        PSVAE_TRY(launch(e));
      } else {
        EpiLatent<TAct> e;
        PSVAE_TRY(launch(e));
      }
      head_done = true;
      if (a.mu) PSVAE_CUDA(cudaMemcpyAsync(a.mu, mu, (size_t)B * n.L * sizeof(float), cudaMemcpyDeviceToDevice, st));
      if (a.ls) PSVAE_CUDA(cudaMemcpyAsync(a.ls, ls, (size_t)B * n.L * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
  }
  if constexpr (sizeof(TAct) == 2) {
    if (grouped_head && !head_done) {
      EpiBiasAct<float, ACT_NONE> e{P + d->enc_b[n.nh], mu, n.L, nullptr};
      PSVAE_TRY((Engine<TAct>::template gemm_grouped<G_FWD>(w.he[n.nh - 1], 2 * n.H, Wt + d->enc_w[n.nh], n.H, B, 2, n.L, n.H, (int64_t)(ls - mu), e, st)));
      head_done = true;
    }
  }
  for (int s = 0; s < 2 && !head_done; ++s) {
    EpiBiasAct<float, ACT_NONE> e{P + d->enc_b[n.nh] + s * n.L, s == 0 ? mu : ls, n.L, nullptr};
    PSVAE_TRY((Engine<TAct>::template gemm<G_FWD>(w.he[n.nh - 1] + s * n.H, 2 * n.H, Wt + d->enc_w[n.nh] + (int64_t)s * n.L * n.H, n.H, B, n.L, n.H, 1, true, e, st)));
  }
  // ---- reparameterisation + KL partial sums (model.py:56-57, lightning.py:115-117) and the latent classifier on mu (lightning.py:73-83,
  //      fp32 on the CUDA cores: C is 2..3).  With linear heads both happen in ONE pass over mu / log_sigma (clf_fused_kernel<REPARAM>).
  const int feat_dim = n.clf_feat();
  const float* feat = mu;
  const bool clf_fused = n.has_clf() && clf_fused_ok(d);
  const bool fuse_latent = clf_fused && a.want_loss;
  int n_kl_used = (int)w.n_kl;
  if (fused_head) {
    n_kl_used = fused_ctas;            // the fused kernel wrote one KL / NLL / accuracy record per CTA
  } else if (!fuse_latent) {
    launch_dep(a.offset_dev ? latent_fwd_kernel<TAct, true> : latent_fwd_kernel<TAct>, dim3((unsigned)w.n_kl), dim3(256), 0, st, mu, ls, a.eps, a.seed,
               a.offset, first_elem, B * n.L, w.z, nullptr, w.kl_part, vae_grads ? w.hs : nullptr, a.offset_dev);
    count_launch();
    PSVAE_LAUNCH_CHECK("latent_fwd_kernel");
  } else {
    // one pass: z, KL partials, logits, CE, accuracy, dlogits, dmu_clf and the classifier's own weight/bias gradients
    ClfFusedArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.n_heads = d->clf_num_heads;
    for (int h = 0; h < d->clf_num_heads; ++h) {
      ca.head_classes[h] = d->clf_head_classes[h];
      ca.head_off[h] = ca.total_classes;
      ca.total_classes += d->clf_head_classes[h];
      ca.w_off[h] = d->clf_head_w[h];
      ca.b_off[h] = d->clf_head_b[h];
    }
    ca.gscale = a.clf_w / ((float)B * (float)d->clf_num_heads);
    ca.write_grad = a.want_grads;
    ca.atomic_out = g_opt.deterministic ? 0 : 1;
    ca.grads = a.want_grads ? a.grads : nullptr;
    ca.sums = w.clf_sums;
    // the classifier's backward moves into the latent backward kernel (fast mode only: it adds with atomics)
    ca.g_rows = (g_opt.clf_grad_in_bwd && vae_grads && ca.atomic_out && w.clf_grows && latent_cs_ok(n.L)) ? w.clf_grows : nullptr;
    const int blocks = clf_fused_blocks(B);
    const size_t smem = clf_fused_smem_bytes(n.L);
    float* dmu_out = vae_grads ? w.dmu_clf : nullptr;
    ReparamArgs rp{ls, a.eps, a.seed, a.offset, first_elem >> 2, w.z, w.kl_part, vae_grads ? w.hs : nullptr, a.offset_dev};
    n_kl_used = blocks;
    switch (n.L) {
#define PSVAE_CLF_CASE(LL)                                                                                                              \
      case LL:                                                                                                                          \
        if (a.offset_dev) PSVAE_TRY((ca.g_rows ? launch_clf_fused<LL, TAct, true, true>(blocks, smem, st, P, mu, a.y, B, ca, dmu_out, w.clf_part, rp)  \
                                               : launch_clf_fused<LL, TAct, false, true>(blocks, smem, st, P, mu, a.y, B, ca, dmu_out, w.clf_part, rp))); \
        else PSVAE_TRY((ca.g_rows ? launch_clf_fused<LL, TAct, true, false>(blocks, smem, st, P, mu, a.y, B, ca, dmu_out, w.clf_part, rp)                 \
                                  : launch_clf_fused<LL, TAct, false, false>(blocks, smem, st, P, mu, a.y, B, ca, dmu_out, w.clf_part, rp)));              \
        break;
      PSVAE_CLF_CASE(16)
      PSVAE_CLF_CASE(32)
      PSVAE_CLF_CASE(64)
      default:
      PSVAE_CLF_CASE(128)
#undef PSVAE_CLF_CASE
    }
    count_launch();
    PSVAE_LAUNCH_CHECK("clf_fused_kernel");
    if (!ca.atomic_out) {
      launch_dep(clf_fused_finish_kernel, dim3((unsigned)ceil_div64(clf_part_len(n.L), 32)), dim3(1024), 0, st, w.clf_part, blocks, n.L, ca, w.clf_sums,
                                                                                             a.want_grads ? a.grads : nullptr);
      count_launch();
      PSVAE_LAUNCH_CHECK("clf_fused_finish_kernel");
    }
  }
  if (fuse_latent || fused_head) {
  } else if (n.has_clf() && a.want_loss) {
    for (int t = 0; t < d->clf_num_trunk; ++t) {
      PSVAE_TRY(clf_linear(d->clf_activation, feat, t == 0 ? n.L : d->clf_hidden, P + d->clf_trunk_w[t], P + d->clf_trunk_b[t], w.clf_act[t], B,
                           d->clf_hidden, n.clf_trunk_in(t), st));
      feat = w.clf_act[t];
    }
    for (int h = 0; h < d->clf_num_heads; ++h) {
      const int C = d->clf_head_classes[h];
      PSVAE_TRY(clf_linear(ACT_NONE, feat, feat_dim, P + d->clf_head_w[h], P + d->clf_head_b[h], w.logits[h], B, C, feat_dim, st));
      const float gscale = a.clf_w / ((float)B * (float)d->clf_num_heads);
      launch_dep(ce_kernel, dim3((unsigned)w.n_ce), dim3(256), 0, st, w.logits[h], a.y + (int64_t)h * B, B, C, gscale, a.want_grads, w.nll_part[h], w.acc_part[h]);
      count_launch();
      PSVAE_LAUNCH_CHECK("ce_kernel");
    }
  }

  // ---- decoder (model.py:58-61) + reconstruction loss (lightning.py:110-113)
  // the consistency term needs x_hat before its gradient can join d loss / d x_hat: it goes through the general (unfused) tail
  const bool general_tail = d->normalize_decoder || a.use_cos || cons_on;
  int n_sse_used = 0;
  bool dec_last_bias_done = false, dec_last_bias_reduce = false;
  if (a.want_loss && !general_tail) {
    const float scale = 2.f / ((float)B * (float)n.D * 10.f);
    bool launched = false;
    int chain_ctas = 0;
    if constexpr (sizeof(TAct) == 2) {
      // option train_chain: the whole decoder + MSE epilogue as one chained kernel (hidden activations stay on-chip for the forward pass)
      if (g_opt.train_chain && vae_grads && !g_opt.deterministic && !a.x_hat && decoder_chain_ok(n.D, n.L, n.H, n.nh) && w.mhd[0] && w.mhd[1]) {
        DcArgs ca;
        memset(&ca, 0, sizeof(ca));
        ca.rows = B; ca.H = n.H; ca.D = n.D;
        ca.b0 = P + d->dec_b[0]; ca.b1 = P + d->dec_b[1]; ca.b2 = P + d->dec_b[2];
        ca.trace = tc_trace_ptr();
        ca.z16 = w.z;
        ca.mask0 = w.mhd[0]; ca.mask1 = w.mhd[1]; ca.mask_ld = B;
        ca.x = a.x16 ? static_cast<const void*>(a.x16) : static_cast<const void*>(a.x);
        ca.x_bf16 = a.x16 ? 1 : 0;
        ca.scale = scale;
        ca.sse_part = w.sse_part;
        ca.bias_grad = a.grads + d->dec_b[n.nh];
        int ctas = 0;
        PSVAE_TRY(decoder_chain_launch<true>(Wt + d->dec_w[0], Wt + d->dec_w[1], Wt + d->dec_w[2], w.dxh, w.hd[0], w.hd[1], ca, st, &ctas));
        launched = dec_last_bias_done = true;
        chain_ctas = ctas;
      }
    }
    if constexpr (sizeof(TAct) == 2) {
      if (!launched && vae_grads && tc_colsum_ok(n.D)) {     // + column sums of dxh = bias gradient of the last decoder layer
        const bool atomic = !g_opt.deterministic;
        if (a.x16) {
          EpiMse<TAct, true, bf16> e{P + d->dec_b[n.nh], a.x16, n.D, a.x_hat, n.D, w.dxh, n.D, scale, w.sse_part, atomic ? a.grads + d->dec_b[n.nh] : w.cpart,
                                     atomic ? 1 : 0};
          PSVAE_TRY(decoder_forward<TAct>(n, Wt, P, w.z, w.hd, B, e, st, (a.want_grads && w.mhd[0]) ? w.mhd : nullptr));
        } else {
          EpiMse<TAct, true> e{P + d->dec_b[n.nh], a.x, n.D, a.x_hat, n.D, w.dxh, n.D, scale, w.sse_part, atomic ? a.grads + d->dec_b[n.nh] : w.cpart,
                               atomic ? 1 : 0};
          PSVAE_TRY(decoder_forward<TAct>(n, Wt, P, w.z, w.hd, B, e, st, (a.want_grads && w.mhd[0]) ? w.mhd : nullptr));
        }
        launched = dec_last_bias_done = true;
        dec_last_bias_reduce = !atomic;
      }
      if (!launched && a.x16) {
        EpiMse<TAct, false, bf16> e{P + d->dec_b[n.nh], a.x16, n.D, a.x_hat, n.D, a.want_grads ? w.dxh : nullptr, n.D, scale, w.sse_part, nullptr, 0};
        PSVAE_TRY(decoder_forward<TAct>(n, Wt, P, w.z, w.hd, B, e, st, (a.want_grads && w.mhd[0]) ? w.mhd : nullptr));
        launched = true;
      }
    }
    if (!launched) {
      EpiMse<TAct> e{P + d->dec_b[n.nh], a.x, n.D, a.x_hat, n.D, a.want_grads ? w.dxh : nullptr, n.D, scale, w.sse_part, nullptr, 0};
      PSVAE_TRY(decoder_forward<TAct>(n, Wt, P, w.z, w.hd, B, e, st, (a.want_grads && w.mhd[0]) ? w.mhd : nullptr));
    }
    n_sse_used = chain_ctas > 0 ? chain_ctas : (sizeof(TAct) == 2 ? (int)tc_ctas(B, n.D, 1, (int)g_opt.tc_force_bn) : (int)sgemm_red_slots(B, n.D));   // one slot per CTA / per tile
    if (dec_last_bias_reduce) PSVAE_TRY(launch_reduce(w.cpart, n.D, n_sse_used * 4, a.grads + d->dec_b[n.nh], st));
  } else {
    float* u = general_tail ? w.u : (a.x_hat ? a.x_hat : w.u);
    EpiBiasAct<float, ACT_NONE> e{P + d->dec_b[n.nh], u, n.D, nullptr};
    PSVAE_TRY(decoder_forward<TAct>(n, Wt, P, w.z, w.hd, B, e, st, (a.want_grads && w.mhd[0]) ? w.mhd : nullptr));
    if (a.ext) {
      // no loss inside: x_hat (if asked for) and d loss / d u from the caller's d loss / d x_hat, through the normalisation when it is on
      const int blocks = (int)ceil_div64(B * 32, 256);
      if (a.ext_gx || (general_tail && a.x_hat)) {
        launch_dep(recon_rows_kernel<TAct>, dim3(blocks), dim3(256), 0, st, u, (const float*)nullptr, B, n.D, d->normalize_decoder, 0, 0.f,
                                                        general_tail ? a.x_hat : (float*)nullptr, a.ext_gx ? w.dxh : (TAct*)nullptr, (float*)nullptr, a.ext_gx);
        count_launch();
        PSVAE_LAUNCH_CHECK("recon_rows_kernel");
      }
      if (!a.ext_gx) PSVAE_CUDA(cudaMemsetAsync(w.dxh, 0, (size_t)B * n.D * sizeof(TAct), st));
    } else if (general_tail) {
      const float gscale = a.use_cos ? 1.f / (float)B : 2.f / ((float)B * (float)n.D * 10.f);
      const int blocks = (int)ceil_div64(B * 32, 256);
      const float* gx = nullptr;
      if (cons_on) {
        // x_hat first (a pass of its own only when it differs from u), then CE(consistency_classifier(x_hat), y) and its gradient w.r.t. x_hat
        const float* xh = w.u;
        if (d->normalize_decoder) {
          float* xh_out = a.x_hat ? a.x_hat : cw.xh;
          launch_dep(recon_rows_kernel<TAct>, dim3(blocks), dim3(256), 0, st, w.u, (const float*)nullptr, B, n.D, 1, 0, 0.f, xh_out, (TAct*)nullptr,
                                                          (float*)nullptr, (const float*)nullptr);
          count_launch();
          PSVAE_LAUNCH_CHECK("recon_rows_kernel");
          xh = xh_out;
        }
        PSVAE_TRY(cons_forward(a.cons, a.cons_params, xh, B, cw, cw.logits, st));
        launch_dep(ce_kernel, dim3((unsigned)cw.n_ce), dim3(256), 0, st, cw.logits, a.cons_y, B, a.cons->num_classes, a.cons_w / (float)B, vae_grads,
                                                cw.nll_part, cw.acc_part);
        count_launch();
        PSVAE_LAUNCH_CHECK("ce_kernel");
        if (vae_grads) {
          PSVAE_TRY(cons_input_grad(a.cons, a.cons_params, B, cw, st));
          gx = cw.gx;
        }
      }
      launch_dep(recon_rows_kernel<TAct>, dim3(blocks), dim3(256), 0, st, w.u, a.want_loss ? a.x : nullptr, B, n.D, d->normalize_decoder, a.use_cos, gscale, a.x_hat,
                                                      vae_grads ? w.dxh : nullptr, a.want_loss ? w.sse_part : nullptr, gx);
      count_launch();
      PSVAE_LAUNCH_CHECK("recon_rows_kernel");
      n_sse_used = blocks;
    }
  }
  // The loss scalars have no consumer on the device: when the backward pass runs the 8-column latent kernel, its last block computes them
  // (one launch boundary less between the forward and the backward pass); otherwise finalize_losses_kernel does, right here.
  LossPartials lp;
  memset(&lp, 0, sizeof(lp));
  bool finalize_in_latent = false;
  if constexpr (sizeof(TAct) == 2) {
    int total_classes = 0;
    for (int h = 0; h < d->clf_num_heads; ++h) total_classes += d->clf_head_classes[h];
    finalize_in_latent = a.want_loss && vae_grads && !a.ext && clf_fused && (g_opt.clf_grad_in_bwd || fused_head) && !g_opt.deterministic &&
                         w.clf_grows && latent_cs_ok(n.L) && latent8_ok(n.L, total_classes);
  }
  if (a.want_loss) {
    lp.sse = w.sse_part; lp.n_sse = n_sse_used;
    lp.kl = w.kl_part; lp.n_kl = n_kl_used;
    const bool ce_from_blocks = clf_fused && !g_opt.deterministic;     // fused pass, fast mode: one (nll, acc) record per block
    lp.n_ce = clf_fused ? (ce_from_blocks ? clf_fused_blocks(B) : 1) : (int)w.n_ce;
    lp.ce_stride = ce_from_blocks ? clf_part_len(n.L) : 1;
    lp.n_heads = n.has_clf() ? d->clf_num_heads : 0;
    for (int h = 0; h < lp.n_heads; ++h) {
      lp.nll[h] = clf_fused ? (ce_from_blocks ? w.clf_part + h : w.clf_sums + h) : w.nll_part[h];
      lp.acc[h] = clf_fused ? (ce_from_blocks ? w.clf_part + 4 + h : w.clf_sums + 4 + h) : w.acc_part[h];
    }
    lp.recon_scale = a.use_cos ? 1.f / (float)B : 1.f / ((float)B * (float)n.D * 10.f);
    lp.inv_b = 1.f / (float)B;
    if (fused_head && lp.n_heads > 0) { lp.nll[0] = w.clf_part; lp.acc[0] = w.clf_part + PSVAE_NUM_SMS; lp.n_ce = fused_ctas; lp.ce_stride = 1; }
    lp.kl_w = a.kl_w; lp.clf_w = a.clf_w;
    if (cons_on) { lp.cons_nll = cw.nll_part; lp.cons_acc = cw.acc_part; lp.n_cons = (int)cw.n_ce; lp.cons_w = a.cons_w; }
    if (!finalize_in_latent) {
      launch_dep(finalize_losses_kernel, dim3(1), dim3(1024), 0, st, lp, a.losses);
      count_launch();
      PSVAE_LAUNCH_CHECK("finalize_losses_kernel");
    }
  }
  if (!a.want_grads) return 0;

  // =================================== backward (SURVEY 3.5) ===================================
  float* G = a.grads;
  w.merge_wgrads = sizeof(TAct) == 2 && g_opt.tc_merged_wgrad && !g_opt.deterministic;
  // a gradient buffer that a collected (not yet launched) wgrad problem reads must not be overwritten: launch what is pending first
  auto before_write = [&](const void* buf) -> int {
    for (int i = 0; i < w.n_pending; ++i)
      if (w.pending[i].dY == buf || static_cast<const char*>(w.pending[i].dY) == static_cast<const char*>(buf) + (size_t)n.H * sizeof(TAct))
        return flush_wgrads(w, B, st);
    return 0;
  };

  // ---- classifier backward -> dmu_clf (the fused kernel already produced it together with the classifier's gradients)
  const float* dmu_clf = (clf_fused && a.want_loss) ? w.dmu_clf : nullptr;
  if (a.ext) dmu_clf = a.ext_gmu;                      // the caller's d loss / d mu takes the classifier gradient's place
  if (n.has_clf() && !clf_fused && a.want_loss) {
    const int T = d->clf_num_trunk;
    const float* featp = T > 0 ? w.clf_act[T - 1] : mu;
    for (int h = 0; h < d->clf_num_heads; ++h) {
      const int C = d->clf_head_classes[h];
      PSVAE_TRY(wgrad_clf<TAct>(w.logits[h], C, featp, feat_dim, B, C, feat_dim, G + d->clf_head_w[h], G + d->clf_head_b[h], w, st));
    }
    if (T == 0) {
      for (int h = 0; h < d->clf_num_heads && vae_grads; ++h)
        PSVAE_TRY(clf_dgrad(ACT_NONE, w.logits[h], d->clf_head_classes[h], P + d->clf_head_w[h], n.L, nullptr, w.dmu_clf, h > 0 ? 1.f : 0.f, B, st));
    } else {
      float* cur = w.clf_g[0];
      float* nxt = w.clf_g[1];
      for (int h = 0; h < d->clf_num_heads; ++h)   // dU_{T-1} = sum_h (dlogits_h W_h) .* act'(A_{T-1})
        PSVAE_TRY(clf_dgrad(d->clf_activation, w.logits[h], d->clf_head_classes[h], P + d->clf_head_w[h], d->clf_hidden, w.clf_act[T - 1], cur,
                            h > 0 ? 1.f : 0.f, B, st));
      for (int t = T - 1; t >= 0; --t) {
        const float* ain = t == 0 ? mu : w.clf_act[t - 1];
        const int in_dim = n.clf_trunk_in(t);
        PSVAE_TRY(wgrad_clf<TAct>(cur, d->clf_hidden, ain, in_dim, B, d->clf_hidden, in_dim, G + d->clf_trunk_w[t], G + d->clf_trunk_b[t], w, st));
        if (t > 0) {
          PSVAE_TRY(clf_dgrad(d->clf_activation, cur, d->clf_hidden, P + d->clf_trunk_w[t], in_dim, w.clf_act[t - 1], nxt, 0.f, B, st));
          float* tmp = cur; cur = nxt; nxt = tmp;
        } else if (vae_grads) {       // the classifier scope stops at the trunk's first layer: d loss / d mu has no consumer
          PSVAE_TRY(clf_dgrad(ACT_NONE, cur, d->clf_hidden, P + d->clf_trunk_w[0], n.L, nullptr, w.dmu_clf, 0.f, B, st));
        }
      }
    }
    dmu_clf = w.dmu_clf;
  }
  if (clf_only) {
    // linear heads: the fused classifier pass (+ its finish kernel) already wrote the gradients, except under the fused encoder head, which
    // leaves d loss / d logits per row in clf_grows (the full step folds them into the latent backward)
    if (!fused_head) return 0;
    if (!latent_cs_ok(n.L)) { set_error("classifier scope: latent_dim=%d has no row-gradient kernel", n.L); return -2; }
    ClfBwdArgs cb;
    memset(&cb, 0, sizeof(cb));
    cb.n_heads = d->clf_num_heads;
    for (int h = 0; h < d->clf_num_heads; ++h) {
      cb.head_classes[h] = d->clf_head_classes[h];
      cb.head_off[h] = cb.total_classes;
      cb.total_classes += d->clf_head_classes[h];
      cb.w_off[h] = d->clf_head_w[h];
      cb.b_off[h] = d->clf_head_b[h];
    }
    cb.params = P; cb.grads = G; cb.g_rows = w.clf_grows;
    int blocks = ew_grid(B * n.L / 4);
    if (blocks > 2 * PSVAE_NUM_SMS) blocks = 2 * PSVAE_NUM_SMS;      // 8 blocks per SM measured slower: more atomics on the same 130 floats
    if (cb.total_classes <= 4) launch_dep(clf_rows_wgrad_kernel<4>, dim3(blocks), dim3(256), 0, st, (const float*)mu, B * n.L, n.L, cb);
    else launch_dep(clf_rows_wgrad_kernel<CLF_MAXC>, dim3(blocks), dim3(256), 0, st, (const float*)mu, B * n.L, n.L, cb);
    count_launch();
    PSVAE_LAUNCH_CHECK("clf_rows_wgrad_kernel");
    return 0;
  }

  // ---- decoder backward: dY starts as d loss / d (decoder output)
  {
    const TAct* dY = w.dxh;
    int out_dim = n.D;
    int pp = 0;
    bool bias_done = dec_last_bias_done;
    for (int j = n.nh; j >= 0; --j) {
      const TAct* ain = j == 0 ? w.z : w.hd[j - 1];
      const int in_dim = n.dec_in(j);
      PSVAE_TRY(wgrad<TAct>(dY, out_dim, ain, in_dim, B, out_dim, in_dim, G + d->dec_w[j], bias_done ? nullptr : G + d->dec_b[j], w, st));
      if (j > 0) {
        PSVAE_TRY(before_write(w.gd[pp]));
        PSVAE_TRY(dgrad_hidden<TAct>(dY, out_dim, Wt + d->dec_w[j], out_dim, in_dim, w.hd[j - 1], n.H, w.mhd[j - 1], w.gd[pp], n.H, B,
                                     G + d->dec_b[j - 1], w, &bias_done, st));
        dY = w.gd[pp];
        out_dim = n.H;
        pp ^= 1;
      } else {
        EpiStore e{w.dz, n.L, 0, 1.f, 0.f, nullptr, 0};
        PSVAE_TRY((Engine<TAct>::template gemm<G_DGRAD>(dY, out_dim, Wt + d->dec_w[0], n.L, B, n.L, out_dim, 1, true, e, st)));
      }
    }
  }
  // ---- through the reparameterisation and the KL term (+ the bias gradients of the encoders' last Linear)
  bool last_bias_done = false;
  const bool clf_in_bwd = !a.ext && clf_fused && a.want_loss && (g_opt.clf_grad_in_bwd || fused_head) && !g_opt.deterministic && w.clf_grows && latent_cs_ok(n.L);
  if (clf_in_bwd) {
    int blocks = ew_grid(B * n.L / 4);
    if (blocks > 3 * PSVAE_NUM_SMS) blocks = 3 * PSVAE_NUM_SMS;      // 80 registers x 256 threads: three blocks per SM are resident -- one full wave
    ClfBwdArgs cb;
    memset(&cb, 0, sizeof(cb));
    cb.n_heads = d->clf_num_heads;
    for (int h = 0; h < d->clf_num_heads; ++h) {
      cb.head_classes[h] = d->clf_head_classes[h];
      cb.head_off[h] = cb.total_classes;
      cb.total_classes += d->clf_head_classes[h];
      cb.w_off[h] = d->clf_head_w[h];
      cb.b_off[h] = d->clf_head_b[h];
    }
    cb.params = P; cb.grads = G; cb.g_rows = w.clf_grows;
    const size_t smem = 256 * 8 * sizeof(float);
    float* bias_grad = G + d->enc_b[n.nh];
    bool done8 = false;
    if constexpr (sizeof(TAct) == 2) {
      // the 8-columns-per-thread form: L a multiple of 8 with L / 8 dividing 256, at most 4 classes
      if (latent8_ok(n.L, cb.total_classes)) {
        const int rpb = 256 / (n.L / 8);
        int64_t nb = ceil_div64(B, rpb);
        if (nb > 2 * PSVAE_NUM_SMS) nb = 2 * PSVAE_NUM_SMS;
        if (nb < 1) nb = 1;
#define PSVAE_LBC8(NCV)                                                                                                                       \
        launch_dep(latent_bwd_clf8_kernel<NCV>, dim3((unsigned)nb + (finalize_in_latent ? 1u : 0u)), dim3(256), smem + (size_t)NCV * n.L * sizeof(float), st, w.dz, mu, ls, \
                   w.hs, B, n.L, a.kl_w / (float)B, w.dmu, w.dls, bias_grad, (int64_t)2 * n.L, cb, lp, finalize_in_latent ? a.losses : (float*)nullptr)
        if (cb.total_classes <= 2) PSVAE_LBC8(2);
        else PSVAE_LBC8(4);
#undef PSVAE_LBC8
        done8 = true;
      }
    }
#define PSVAE_LBC(NCV)                                                                                                                          \
    launch_dep(latent_bwd_clf_kernel<TAct, NCV>, dim3(blocks), dim3(256), smem, st, w.dz, mu, ls, w.hs, B * n.L, n.L, a.kl_w / (float)B, w.dmu, w.dls, \
               bias_grad, (int64_t)2 * n.L, cb)
    if (done8) {}
    else if (cb.total_classes <= 2) PSVAE_LBC(2);
    else if (cb.total_classes == 3) PSVAE_LBC(3);
    else PSVAE_LBC(CLF_MAXC);
#undef PSVAE_LBC
    count_launch();
    PSVAE_LAUNCH_CHECK("latent_bwd_clf_kernel");
    last_bias_done = true;
  } else if (latent_cs_ok(n.L)) {
    int blocks = ew_grid(B * n.L / 4);
    if (blocks > 4 * PSVAE_NUM_SMS) blocks = 4 * PSVAE_NUM_SMS;
    float* bias_atomic = g_opt.deterministic ? nullptr : G + d->enc_b[n.nh];      // fast mode: atomics into the zeroed gradient, no reduce launch
    launch_dep(latent_bwd_cs_kernel<TAct>, dim3(blocks), dim3(256), 256 * 8 * sizeof(float), st, w.dz, mu, ls, w.hs, B * n.L, n.L, dmu_clf,
                                                                             a.kl_w / (float)B, w.dmu, w.dls, w.cpart, bias_atomic, (int64_t)2 * n.L, a.ext ? a.ext_gls : (const float*)nullptr);
    count_launch();
    PSVAE_LAUNCH_CHECK("latent_bwd_cs_kernel");
    if (!bias_atomic) PSVAE_TRY(launch_reduce(w.cpart, 2 * n.L, blocks, G + d->enc_b[n.nh], st));
    last_bias_done = true;
  } else {
    launch_dep(latent_bwd_kernel<TAct>, dim3(ew_grid(B * n.L / 4)), dim3(256), 0, st, w.dz, mu, ls, w.hs, B * n.L, dmu_clf, a.kl_w / (float)B,
                                                                  w.dmu, w.dls, n.L / 4, (int64_t)2 * n.L, a.ext ? a.ext_gls : (const float*)nullptr);
    count_launch();
    PSVAE_LAUNCH_CHECK("latent_bwd_kernel");
  }

  // ---- encoders backward
  {
    int pp = 0;
    bool bias_done[2] = {false, false};
    // grouped dgrad of both encoders' layer j (tcgen05 mode): dY [B][2 Kg] x stacked W [2 Kg][H] -> [B][2H] .* ReLU' (+ bias gradient of layer j-1)
    auto dgrad_pair = [&](const TAct* dY, int64_t ldy, int Kg, int layer, TAct* out) -> int {
      if constexpr (sizeof(TAct) == 2) {
        const bool atomic = !g_opt.deterministic;
        EpiActGrad<TAct, TAct, ACT_RELU, true> e{w.he[layer - 1], 2 * n.H, w.mhe[layer - 1], B, out, 2 * n.H, 0.f, nullptr,
                                                 atomic ? G + d->enc_b[layer - 1] : w.cpart, atomic ? 1 : 0};
        PSVAE_TRY((Engine<TAct>::template gemm_grouped<G_DGRAD>(dY, ldy, Wt + d->enc_w[layer], n.H, B, 2, n.H, Kg, 0, e, st)));
        if (!atomic) {
          // the grouped launch tiles by ONE group's width (a tile never straddles the two encoders): count its CTAs with that tile width
          const int bn_g = g_opt.tc_force_bn ? (int)g_opt.tc_force_bn : tc_pick_bn(n.H);
          const int64_t ctas = tc_ctas(B, 2 * n.H, 1, bn_g);
          PSVAE_TRY(launch_reduce(w.cpart, 2 * n.H, (int)ctas * 4, G + d->enc_b[layer - 1], st));
        }
        bias_done[0] = bias_done[1] = true;
      }
      return 0;
    };
    const int64_t ld_lat = 2 * n.L;      // dmu | dls share one [B][2L] buffer
    // last layer (mu / sigma heads): wgrad per encoder, dgrad grouped where it can be
    for (int s = 0; s < 2; ++s) {
      const TAct* dY = s == 0 ? w.dmu : w.dls;
      PSVAE_TRY(wgrad<TAct>(dY, ld_lat, w.he[n.nh - 1] + s * n.H, 2 * n.H, B, n.L, n.H, G + d->enc_w[n.nh] + (int64_t)s * n.L * n.H,
                            last_bias_done ? nullptr : G + d->enc_b[n.nh] + s * n.L, w, st));
    }
    bool head_grouped = false;
    if constexpr (sizeof(TAct) == 2) {
      if (Engine<TAct>::grouped_ok(n.H, n.L) && w.mhe[n.nh - 1] && tc_colsum_ok(n.H)) {
        PSVAE_TRY(dgrad_pair(w.dmu, ld_lat, n.L, n.nh, w.ge[pp]));
        head_grouped = true;
      }
    }
    for (int s = 0; s < 2 && !head_grouped; ++s) {
      const TAct* dY = s == 0 ? w.dmu : w.dls;
      PSVAE_TRY(dgrad_hidden<TAct>(dY, ld_lat, Wt + d->enc_w[n.nh] + (int64_t)s * n.L * n.H, n.L, n.H, w.he[n.nh - 1] + s * n.H, 2 * n.H,
                                   w.mhe[n.nh - 1] ? w.mhe[n.nh - 1] + (int64_t)s * (n.H / 32) * B : nullptr, w.ge[pp] + s * n.H, 2 * n.H, B,
                                   G + d->enc_b[n.nh - 1] + s * n.H, w, &bias_done[s], st));
    }
    for (int j = n.nh - 1; j >= 1; --j) {
      for (int s = 0; s < 2; ++s) {
        const TAct* dY = w.ge[pp] + s * n.H;
        PSVAE_TRY(wgrad<TAct>(dY, 2 * n.H, w.he[j - 1] + s * n.H, 2 * n.H, B, n.H, n.H, G + d->enc_w[j] + (int64_t)s * n.H * n.H,
                              bias_done[s] ? nullptr : G + d->enc_b[j] + s * n.H, w, st));
      }
      bool pair_done = false;
      PSVAE_TRY(before_write(w.ge[pp ^ 1]));
      if constexpr (sizeof(TAct) == 2) {
        if (grouped_hidden && w.mhe[j - 1] && tc_colsum_ok(n.H)) {
          PSVAE_TRY(dgrad_pair(w.ge[pp], 2 * n.H, n.H, j, w.ge[pp ^ 1]));
          pair_done = true;
        }
      }
      for (int s = 0; s < 2 && !pair_done; ++s) {
        const TAct* dY = w.ge[pp] + s * n.H;
        PSVAE_TRY(dgrad_hidden<TAct>(dY, 2 * n.H, Wt + d->enc_w[j] + (int64_t)s * n.H * n.H, n.H, n.H, w.he[j - 1] + s * n.H, 2 * n.H,
                                     w.mhe[j - 1] ? w.mhe[j - 1] + (int64_t)s * (n.H / 32) * B : nullptr, w.ge[pp ^ 1] + s * n.H, 2 * n.H, B,
                                     G + d->enc_b[j - 1] + s * n.H, w, &bias_done[s], st));
      }
      pp ^= 1;
    }
    // layer 0: both encoders in one wgrad ([2H, D]); x needs no gradient (SURVEY 3.5)
    if (bias_done[0] && bias_done[1]) {
      PSVAE_TRY(wgrad<TAct>(w.ge[pp], 2 * n.H, xa, n.D, B, 2 * n.H, n.D, G + d->enc_w[0], nullptr, w, st));
    } else {
      PSVAE_TRY(wgrad<TAct>(w.ge[pp], 2 * n.H, xa, n.D, B, 2 * n.H, n.D, G + d->enc_w[0], G + d->enc_b[0], w, st));
    }
  }
  return flush_wgrads(w, B, st);
}

// ------------------------------------------------------------------------------------------------
// decode / sampling
// ------------------------------------------------------------------------------------------------
template <typename TAct>
static int run_decode(const psvae_model_desc* d, const float* params, const bf16* shadow, const float* z, uint64_t seed, uint64_t offset, int64_t row0,
                      int64_t rows, float* x_hat, float* z_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
  PSVAE_TRY(tc_device_check());
  Net n(d);
  if (rows <= 0) { set_error("rows=%lld must be positive", (long long)rows); return -2; }
  if (!params || !x_hat) { set_error("params and x_hat must not be NULL"); return -1; }
  if (sizeof(TAct) == 2 && !shadow) { set_error("PSVAE_BF16 needs the bf16 shadow copy of the parameters (psvae_refresh_shadow)"); return -1; }
  if constexpr (sizeof(TAct) == 2) {
    // the chained kernel: no scratch, no chunking -- every hidden activation stays on the SM that produced it
    if (g_opt.decode_chain && !d->normalize_decoder && decoder_chain_ok(n.D, n.L, n.H, n.nh) && (reinterpret_cast<uintptr_t>(x_hat) & 15) == 0 &&
        (!z || (reinterpret_cast<uintptr_t>(z) & 15) == 0) && (!z_out || (reinterpret_cast<uintptr_t>(z_out) & 15) == 0)) {
      DcArgs a;
      memset(&a, 0, sizeof(a));
      a.rows = rows; a.H = n.H; a.D = n.D;
      a.b0 = params + d->dec_b[0]; a.b1 = params + d->dec_b[1]; a.b2 = params + d->dec_b[2];
      a.z_in = z; a.z_out = (z_out && z_out != z) ? z_out : nullptr;
      a.seed = seed; a.offset = offset; a.first_row = row0;
      a.trace = tc_trace_ptr();
      return decoder_chain_launch<false>(shadow + d->dec_w[0], shadow + d->dec_w[1], shadow + d->dec_w[2], x_hat, nullptr, nullptr, a, st);
    }
  }
  const int64_t chunk = rows < g_opt.decode_chunk ? rows : g_opt.decode_chunk;
  StepBufs<TAct> w;
  {
    Bump sz(nullptr);
    StepBufs<TAct> tmp;
    plan<TAct>(d, chunk, PSVAE_MODE_DECODE, sz, tmp);
    if (sz.used > ws_bytes || !ws) {
      set_error("workspace too small: need %lld bytes, got %lld", (long long)sz.used, (long long)ws_bytes);
      return -2;
    }
    Bump b(ws);
    plan<TAct>(d, chunk, PSVAE_MODE_DECODE, b, w);
  }
  const TAct* Wt;
  if constexpr (sizeof(TAct) == 2) Wt = shadow; else Wt = params;
  for (int64_t r0 = 0; r0 < rows; r0 += chunk) {
    const int64_t m = rows - r0 < chunk ? rows - r0 : chunk;
    const int64_t nel = m * n.L;
    const TAct* zin;
    if (z) {
      if constexpr (sizeof(TAct) == 2) {
        launch_dep(cast_bf16_kernel, dim3(ew_grid(nel / 8)), dim3(256), 0, st, z + r0 * n.L, w.z, nel, (float*)nullptr, (int64_t)0);
        count_launch();
        PSVAE_LAUNCH_CHECK("cast_bf16_kernel");
        zin = w.z;
      } else {
        zin = z + r0 * n.L;
      }
      if (z_out && z_out != z) PSVAE_CUDA(cudaMemcpyAsync(z_out + r0 * n.L, z + r0 * n.L, (size_t)nel * sizeof(float), cudaMemcpyDeviceToDevice, st));
    } else {
      const int64_t first = (row0 + r0) * n.L;
      if (z_out) {
        launch_dep(philox_normal_kernel<float>, dim3(ew_grid(nel / 4)), dim3(256), 0, st, z_out + r0 * n.L, nel, seed, offset, first);
        count_launch();
        PSVAE_LAUNCH_CHECK("philox_normal_kernel");
        if constexpr (sizeof(TAct) == 2) {
          launch_dep(cast_bf16_kernel, dim3(ew_grid(nel / 8)), dim3(256), 0, st, z_out + r0 * n.L, w.z, nel, (float*)nullptr, (int64_t)0);
          count_launch();
          PSVAE_LAUNCH_CHECK("cast_bf16_kernel");
          zin = w.z;
        } else {
          zin = z_out + r0 * n.L;
        }
      } else {
        launch_dep(philox_normal_kernel<TAct>, dim3(ew_grid(nel / 4)), dim3(256), 0, st, w.z, nel, seed, offset, first);
        count_launch();
        PSVAE_LAUNCH_CHECK("philox_normal_kernel");
        zin = w.z;
      }
    }
    float* out = x_hat + r0 * n.D;
    EpiBiasAct<float, ACT_NONE> e{params + d->dec_b[n.nh], out, n.D, nullptr};
    PSVAE_TRY(decoder_forward<TAct>(n, Wt, params, zin, w.hd, m, e, st));
    if (d->normalize_decoder) {
      launch_dep(row_normalize_kernel, dim3((unsigned)ceil_div64(m * 32, 256)), dim3(256), 0, st, out, m, n.D);
      count_launch();
      PSVAE_LAUNCH_CHECK("row_normalize_kernel");
    }
  }
  return 0;
}

}  // namespace psvae

// =================================================================================================
// extern "C"
// =================================================================================================
using namespace psvae;

extern "C" {

int psvae_abi_version(void) { return PSVAE_ABI_VERSION; }
const char* psvae_last_error_string(void) { return g_err; }
int64_t psvae_launch_count(void) { return g_launches.load(); }

int psvae_set_option(const char* name, int64_t value) {
  if (!name) { set_error("option name is NULL"); return -1; }
  if (!strcmp(name, "decode_chunk")) { if (value < 128) value = 128; g_opt.decode_chunk = value; return 0; }
  if (!strcmp(name, "wgrad_split_cap")) { if (value < 1) value = 1; g_opt.wgrad_split_cap = value; return 0; }
  if (!strcmp(name, "colsum_rows")) { if (value < 8) value = 8; g_opt.colsum_rows = value; return 0; }
  if (!strcmp(name, "tc_force_bn")) {
    if (value != 0 && value != 64 && value != 128 && value != 256) { set_error("tc_force_bn must be 0, 64, 128 or 256"); return -2; }
    g_opt.tc_force_bn = value; return 0;
  }
  if (!strcmp(name, "tc_grid_limit")) { g_opt.tc_grid_limit = value < 0 ? 0 : value; return 0; }
  if (!strcmp(name, "deterministic")) { g_opt.deterministic = value ? 1 : 0; return 0; }
  if (!strcmp(name, "tc_two_cta")) { g_opt.tc_two_cta = value ? 1 : 0; return 0; }
  if (!strcmp(name, "langevin_generic")) { g_opt.langevin_generic = value ? 1 : 0; return 0; }
  if (!strcmp(name, "tc_max_stages")) { g_opt.tc_max_stages = value < 0 ? 0 : value; return 0; }
  if (!strcmp(name, "tc_trace_ptr")) { g_opt.tc_trace_ptr = value; return 0; }
  if (!strcmp(name, "tc_trace_skip")) { g_opt.tc_trace_skip = value; g_opt.tc_trace_select = 1; return 0; }
  if (!strcmp(name, "tc_trace_select")) { g_opt.tc_trace_select = value ? 1 : 0; if (!value) g_opt.tc_trace_skip = 0; return 0; }
  if (!strcmp(name, "pdl")) { g_opt.pdl = value ? 1 : 0; return 0; }
  if (!strcmp(name, "tc_grouped")) { g_opt.tc_grouped = value ? 1 : 0; return 0; }
  if (!strcmp(name, "tc_epi_groups")) { g_opt.tc_epi_groups = value ? 1 : 0; return 0; }
  if (!strcmp(name, "wgrad_order")) { g_opt.wgrad_order = value; return 0; }
  if (!strcmp(name, "tc_bn_rounds")) { g_opt.tc_bn_rounds = value ? 1 : 0; return 0; }
  if (!strcmp(name, "wgrad_splits")) { g_opt.wgrad_splits = value < 0 ? 0 : value; return 0; }
  if (!strcmp(name, "tc_epi_groups_max_k")) { g_opt.tc_epi_groups_max_k = value < 0 ? 0 : value; return 0; }
  if (!strcmp(name, "clf_grad_in_bwd")) { g_opt.clf_grad_in_bwd = value ? 1 : 0; return 0; }
  if (!strcmp(name, "fused_head")) { g_opt.fused_head = value ? 1 : 0; return 0; }
  if (!strcmp(name, "tc_merged_wgrad")) { g_opt.tc_merged_wgrad = value ? 1 : 0; return 0; }
  if (!strcmp(name, "decode_chain")) { g_opt.decode_chain = value ? 1 : 0; return 0; }
  if (!strcmp(name, "train_chain")) { g_opt.train_chain = value ? 1 : 0; return 0; }
  if (!strcmp(name, "topk_key_splits")) { g_opt.topk_key_splits = value < 0 ? 0 : value; return 0; }
  set_error("unknown option '%s'", name);
  return -2;
}
int64_t psvae_get_option(const char* name) {
  if (!name) return -1;
  if (!strcmp(name, "decode_chunk")) return g_opt.decode_chunk;
  if (!strcmp(name, "wgrad_split_cap")) return g_opt.wgrad_split_cap;
  if (!strcmp(name, "colsum_rows")) return g_opt.colsum_rows;
  if (!strcmp(name, "tc_force_bn")) return g_opt.tc_force_bn;
  if (!strcmp(name, "tc_grid_limit")) return g_opt.tc_grid_limit;
  if (!strcmp(name, "deterministic")) return g_opt.deterministic;
  if (!strcmp(name, "tc_two_cta")) return g_opt.tc_two_cta;
  if (!strcmp(name, "langevin_generic")) return g_opt.langevin_generic;
  if (!strcmp(name, "tc_max_stages")) return g_opt.tc_max_stages;
  if (!strcmp(name, "pdl")) return g_opt.pdl;
  if (!strcmp(name, "tc_grouped")) return g_opt.tc_grouped;
  if (!strcmp(name, "tc_epi_groups")) return g_opt.tc_epi_groups;
  if (!strcmp(name, "wgrad_order")) return g_opt.wgrad_order;
  if (!strcmp(name, "tc_bn_rounds")) return g_opt.tc_bn_rounds;
  if (!strcmp(name, "wgrad_splits")) return g_opt.wgrad_splits;
  if (!strcmp(name, "tc_epi_groups_max_k")) return g_opt.tc_epi_groups_max_k;
  if (!strcmp(name, "clf_grad_in_bwd")) return g_opt.clf_grad_in_bwd;
  if (!strcmp(name, "fused_head")) return g_opt.fused_head;
  if (!strcmp(name, "tc_merged_wgrad")) return g_opt.tc_merged_wgrad;
  if (!strcmp(name, "decode_chain")) return g_opt.decode_chain;
  if (!strcmp(name, "train_chain")) return g_opt.train_chain;
  if (!strcmp(name, "topk_key_splits")) return g_opt.topk_key_splits;
  return -1;
}

int psvae_model_desc_init(psvae_model_desc* desc, int32_t input_dim, int32_t latent_dim, int32_t hidden_dim, int32_t num_hidden,
                          int32_t normalize_decoder, int32_t clf_num_trunk, int32_t clf_hidden, int32_t clf_activation, int32_t clf_num_heads,
                          int32_t clf_single_label, const int32_t* clf_head_classes) {
  if (!desc) { set_error("desc is NULL"); return -1; }
  memset(desc, 0, sizeof(*desc));
  desc->input_dim = input_dim; desc->latent_dim = latent_dim; desc->hidden_dim = hidden_dim; desc->num_hidden = num_hidden;
  desc->normalize_decoder = normalize_decoder ? 1 : 0;
  desc->clf_num_trunk = clf_num_trunk; desc->clf_hidden = clf_hidden; desc->clf_activation = clf_activation;
  desc->clf_num_heads = clf_num_heads; desc->clf_single_label = clf_single_label ? 1 : 0;
  if (clf_num_heads > 0 && clf_num_heads <= PSVAE_MAX_CLF_HEADS) {
    if (!clf_head_classes) { set_error("clf_head_classes is NULL"); return -1; }
    for (int h = 0; h < clf_num_heads; ++h) desc->clf_head_classes[h] = clf_head_classes[h];
  }
  PSVAE_TRY(check_desc(desc, PSVAE_FP32));
  Net n(desc);
  int64_t off = 0;
  auto put = [&](int64_t numel) { const int64_t o = off; off = align_up64(off + numel, 8); return o; };
  for (int j = 0; j <= n.nh; ++j) {
    desc->enc_w[j] = put(2ll * n.enc_out(j) * n.enc_in(j));
    desc->enc_b[j] = put(2ll * n.enc_out(j));
  }
  for (int j = 0; j <= n.nh; ++j) {
    desc->dec_w[j] = put((int64_t)n.dec_out(j) * n.dec_in(j));
    desc->dec_b[j] = put(n.dec_out(j));
  }
  desc->vae_numel = off;
  if (clf_num_heads > 0) {
    for (int t = 0; t < clf_num_trunk; ++t) {
      desc->clf_trunk_w[t] = put((int64_t)clf_hidden * n.clf_trunk_in(t));
      desc->clf_trunk_b[t] = put(clf_hidden);
    }
    for (int h = 0; h < clf_num_heads; ++h) {
      desc->clf_head_w[h] = put((int64_t)desc->clf_head_classes[h] * n.clf_feat());
      desc->clf_head_b[h] = put(desc->clf_head_classes[h]);
    }
  }
  desc->total_numel = align_up64(off, 64);
  return 0;
}

int64_t psvae_workspace_bytes(const psvae_model_desc* desc, int64_t rows, int32_t precision, int32_t mode) {
  if (check_desc(desc, precision) != 0) return -1;
  if (rows <= 0 || mode < 0 || mode > PSVAE_MODE_TRAIN_CLASSIFIER) { set_error("bad rows/mode"); return -1; }
  if (mode == PSVAE_MODE_DECODE && rows > g_opt.decode_chunk) rows = g_opt.decode_chunk;
  Bump b(nullptr);
  if (precision == PSVAE_BF16) { StepBufs<bf16> w; plan<bf16>(desc, rows, mode, b, w); }
  else { StepBufs<float> w; plan<float>(desc, rows, mode, b, w); }
  return b.used + 256;
}
int64_t psvae_shadow_bytes(const psvae_model_desc* desc) { return desc ? desc->total_numel * (int64_t)sizeof(bf16) : -1; }

int64_t psvae_flops_per_sample(const psvae_model_desc* desc, int32_t mode) {
  if (!desc) return -1;
  Net n(desc);
  int64_t enc = 0, enc_first = 0, dec = 0;
  for (int j = 0; j <= n.nh; ++j) {
    enc += 2ll * n.enc_out(j) * n.enc_in(j);
    dec += (int64_t)n.dec_out(j) * n.dec_in(j);
  }
  enc_first = 2ll * n.enc_out(0) * n.enc_in(0);
  int64_t clf = 0;
  if (n.has_clf()) {
    for (int t = 0; t < desc->clf_num_trunk; ++t) clf += (int64_t)desc->clf_hidden * n.clf_trunk_in(t);
    for (int h = 0; h < desc->clf_num_heads; ++h) clf += (int64_t)desc->clf_head_classes[h] * n.clf_feat();
  }
  if (mode == 2) return 2 * dec;
  if (mode == 1) return 2 * (enc + dec);
  // train: forward + wgrad (same MACs as forward) + dgrad (forward minus the encoders' first layers); classifier fwd + wgrad + dgrad
  return 2 * ((enc + dec) * 3 - enc_first + 3 * clf);
}

// The Adam update behind every psvae_adam_step* entry point.  dc: the device-counter form (lr_dev, counters), else the host form (lr, step).
// Without amsgrad and maximize the pass reads float4: the buffers must be 16-byte aligned.
static int adam_update(bool dc, float* p, const float* g, float* m, float* v, float* vmax, int64_t n, double lr, int64_t step, const double* lr_dev,
                       const psvae_step_counters* counters, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                       int32_t amsgrad, int32_t maximize, int32_t clip_mode, const float* clip_coef, double clip_value, void* shadow_bf16,
                       void* stream) {
  PSVAE_TRY(tc_device_check());
  if (clip_mode != PSVAE_CLIP_NONE && clip_mode != PSVAE_CLIP_NORM && clip_mode != PSVAE_CLIP_VALUE) {
    set_error("clip_mode=%d is not a PSVAE_CLIP_* value", (int)clip_mode);
    return -2;
  }
  if (!p || !g || !m || !v || (amsgrad && !vmax) || (dc && (!lr_dev || !counters)) || (clip_mode == PSVAE_CLIP_NORM && !clip_coef)) {
    set_error("p, g, m, v (vmax with amsgrad, lr and counters in the device-counter form, clip_coef with PSVAE_CLIP_NORM) must not be NULL");
    return -1;
  }
  if (clip_mode == PSVAE_CLIP_VALUE && !(clip_value >= 0.0)) { set_error("clip_value=%g must be >= 0", clip_value); return -2; }
  if (n <= 0) return 0;
  if (!dc && step < 1) { set_error("step=%lld must be >= 1 (count after increment)", (long long)step); return -2; }
  const bool ex = amsgrad || maximize;
  if (!ex && ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) != 0) {
    set_error("Adam buffers must be 16-byte aligned");
    return -2;
  }
  AdamArgs a;
  if (dc) {                  // formed on the device from *lr_dev and the step counter
    a.lr_step = 0.f; a.bc2_sqrt = 1.f;
  } else {
    // host scalars exactly as torch's single-tensor Adam computes them: in python doubles, each rounded to fp32 once where
    // the tensor op consumes it (torch/optim/adam.py:476-547)
    const double bc1 = 1.0 - pow(beta1, (double)step);
    const double bc2 = 1.0 - pow(beta2, (double)step);
    a.lr_step = (float)(lr / bc1);
    a.bc2_sqrt = (float)sqrt(bc2);
  }
  a.beta1 = (float)beta1; a.beta2 = (float)beta2;
  a.one_minus_beta1 = (float)(1.0 - beta1);
  a.one_minus_beta2 = (float)(1.0 - beta2);
  a.eps = (float)eps; a.weight_decay = (float)weight_decay; a.grad_scale = (float)grad_scale;
  static_assert(CLIP_NONE == PSVAE_CLIP_NONE && CLIP_NORM == PSVAE_CLIP_NORM && CLIP_VALUE == PSVAE_CLIP_VALUE, "kernels[dc][ex][clip_mode]");
  static decltype(&adam_kernel<false, false, CLIP_NONE>) const kernels[2][2][3] = {
      {{adam_kernel<false, false, CLIP_NONE>, adam_kernel<false, false, CLIP_NORM>, adam_kernel<false, false, CLIP_VALUE>},
       {adam_kernel<false, true, CLIP_NONE>, adam_kernel<false, true, CLIP_NORM>, adam_kernel<false, true, CLIP_VALUE>}},
      {{adam_kernel<true, false, CLIP_NONE>, adam_kernel<true, false, CLIP_NORM>, adam_kernel<true, false, CLIP_VALUE>},
       {adam_kernel<true, true, CLIP_NONE>, adam_kernel<true, true, CLIP_NORM>, adam_kernel<true, true, CLIP_VALUE>}}};
  launch_dep(kernels[dc][ex][clip_mode], dim3(ew_grid(ex ? n : n / 4 + 1)), dim3(256), 0, static_cast<cudaStream_t>(stream), p, g, m, v, vmax, n, a,
             beta1, beta2, lr_dev, dc ? &counters->adam_step : nullptr, (int)amsgrad, (int)maximize, static_cast<bf16*>(shadow_bf16), clip_coef,
             (float)clip_value);
  count_launch();
  PSVAE_LAUNCH_CHECK("adam_kernel");
  return 0;
}

int psvae_adam_step(float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps, double weight_decay,
                    int64_t step, double grad_scale, void* shadow_bf16, void* stream) {
  return adam_update(false, p, g, m, v, nullptr, n, lr, step, nullptr, nullptr, beta1, beta2, eps, weight_decay, grad_scale, 0, 0, PSVAE_CLIP_NONE,
                     nullptr, 0.0, shadow_bf16, stream);
}

int psvae_adam_step_ex(float* p, const float* g, float* m, float* v, float* vmax, int64_t n, double lr, double beta1, double beta2, double eps,
                       double weight_decay, int64_t step, double grad_scale, int32_t amsgrad, int32_t maximize, void* shadow_bf16, void* stream) {
  return adam_update(false, p, g, m, v, vmax, n, lr, step, nullptr, nullptr, beta1, beta2, eps, weight_decay, grad_scale, amsgrad, maximize,
                     PSVAE_CLIP_NONE, nullptr, 0.0, shadow_bf16, stream);
}

int psvae_adam_step_dc(float* p, const float* g, float* m, float* v, float* vmax, int64_t n, const double* lr, const psvae_step_counters* counters,
                       double beta1, double beta2, double eps, double weight_decay, double grad_scale, int32_t amsgrad, int32_t maximize, void* shadow_bf16,
                       void* stream) {
  return adam_update(true, p, g, m, v, vmax, n, 0.0, 0, lr, counters, beta1, beta2, eps, weight_decay, grad_scale, amsgrad, maximize,
                     PSVAE_CLIP_NONE, nullptr, 0.0, shadow_bf16, stream);
}

int psvae_step_counters_advance(psvae_step_counters* counters, void* stream) { return psvae_step_counters_advance_by(counters, 1, 1, stream); }

int psvae_step_counters_advance_by(psvae_step_counters* counters, uint64_t rng_delta, int64_t step_delta, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!counters) { set_error("counters must not be NULL"); return -1; }
  launch_dep(step_counters_advance_by_kernel, dim3(1), dim3(1), 0, static_cast<cudaStream_t>(stream), &counters->rng_offset, &counters->adam_step,
             rng_delta, step_delta);
  count_launch();
  PSVAE_LAUNCH_CHECK("step_counters_advance_by_kernel");
  return 0;
}

int psvae_grad_norm(const float* g, const int64_t* spans, int32_t n_spans, double grad_scale, double max_norm, float* total_norm, float* coef,
                    void* scratch, int64_t scratch_bytes, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!g || !spans || !total_norm || !coef || !scratch) { set_error("g, spans, total_norm, coef and scratch must not be NULL"); return -1; }
  if (n_spans < 1 || n_spans > GRAD_NORM_MAX_SPANS) { set_error("n_spans=%d must be in [1, %d]", (int)n_spans, GRAD_NORM_MAX_SPANS); return -2; }
  if (scratch_bytes < PSVAE_GRAD_NORM_SCRATCH_BYTES || (reinterpret_cast<uintptr_t>(scratch) & 7) != 0) {
    set_error("scratch must be 8-byte aligned and hold PSVAE_GRAD_NORM_SCRATCH_BYTES = %d bytes", PSVAE_GRAD_NORM_SCRATCH_BYTES);
    return -2;
  }
  GradNormSpans sp{};
  sp.n = n_spans;
  for (int i = 0; i < n_spans; ++i) {
    sp.a[i] = spans[2 * i];
    sp.b[i] = spans[2 * i + 1];
    if (sp.a[i] < 0 || sp.b[i] < sp.a[i]) { set_error("span %d = [%lld, %lld) is invalid", i, (long long)sp.a[i], (long long)sp.b[i]); return -2; }
  }
  double* part = static_cast<double*>(scratch);
  unsigned* ticket = reinterpret_cast<unsigned*>(part + GRAD_NORM_BLOCKS);
  launch_dep(grad_norm_kernel, dim3(GRAD_NORM_BLOCKS), dim3(256), 0, static_cast<cudaStream_t>(stream), g, sp, (float)grad_scale, (float)max_norm,
             part, ticket, total_norm, coef);
  count_launch();
  PSVAE_LAUNCH_CHECK("grad_norm_kernel");
  return 0;
}

int psvae_adam_step_clip(float* p, const float* g, float* m, float* v, float* vmax, int64_t n, double lr, int64_t step, const double* lr_dev,
                         const psvae_step_counters* counters, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                         int32_t amsgrad, int32_t maximize, int32_t clip_mode, const float* clip_coef, double clip_value, void* shadow_bf16,
                         void* stream) {
  return adam_update(counters != nullptr, p, g, m, v, vmax, n, lr, step, lr_dev, counters, beta1, beta2, eps, weight_decay, grad_scale, amsgrad,
                     maximize, clip_mode, clip_coef, clip_value, shadow_bf16, stream);
}

int psvae_philox_uint32(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, int64_t first_elem, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!out) { set_error("out is NULL"); return -1; }
  if (n <= 0) return 0;
  launch_dep(philox_u32_kernel, dim3(ew_grid(n / 4 + 1)), dim3(256), 0, static_cast<cudaStream_t>(stream), out, n, seed, offset, first_elem);
  count_launch();
  PSVAE_LAUNCH_CHECK("philox_u32_kernel");
  return 0;
}

int psvae_philox_normal(float* out, int64_t n_rows, int32_t n_cols, uint64_t seed, uint64_t offset, int64_t row0, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!out) { set_error("out is NULL"); return -1; }
  if (n_rows <= 0) return 0;
  if (n_cols <= 0 || n_cols % 4) { set_error("n_cols=%d must be a positive multiple of 4", n_cols); return -2; }
  const int64_t n = n_rows * n_cols;
  launch_dep(philox_normal_kernel<float>, dim3(ew_grid(n / 4)), dim3(256), 0, static_cast<cudaStream_t>(stream), out, n, seed, offset, row0 * n_cols);
  count_launch();
  PSVAE_LAUNCH_CHECK("philox_normal_kernel");
  return 0;
}

int psvae_gather_rows(const void* src, int64_t src_rows, int64_t row_bytes, const int64_t* idx, int64_t n, void* dst, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!src || !idx || !dst) { set_error("src, idx, dst must not be NULL"); return -1; }
  if (n <= 0) return 0;
  if (row_bytes <= 0 || row_bytes % 16 || ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) != 0) {
    set_error("gather: rows must be a multiple of 16 bytes and 16-byte aligned (row_bytes=%lld)", (long long)row_bytes);
    return -2;
  }
  const int vpr = (int)(row_bytes / 16);
  launch_dep(gather_rows_kernel, dim3(ew_grid(n * vpr)), dim3(256), 0, static_cast<cudaStream_t>(stream), static_cast<const uint4*>(src), src_rows, vpr, idx, n,
             static_cast<uint4*>(dst));
  count_launch();
  PSVAE_LAUNCH_CHECK("gather_rows_kernel");
  return 0;
}

int psvae_refresh_shadow(const psvae_model_desc* desc, const float* params, void* shadow_bf16, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!desc || !params || !shadow_bf16) { set_error("desc, params, shadow must not be NULL"); return -1; }
  const int64_t n = desc->total_numel;
  launch_dep(cast_bf16_kernel, dim3(ew_grid(n / 8 + 1)), dim3(256), 0, static_cast<cudaStream_t>(stream), params, static_cast<bf16*>(shadow_bf16), n,
             (float*)nullptr, (int64_t)0);
  count_launch();
  PSVAE_LAUNCH_CHECK("cast_bf16_kernel");
  return 0;
}

// The StepArgs of a model step with what every step takes; x arrives as fp32 or (PSVAE_X_BF16) bf16.  Losses, labels and gradients are off.
static int make_step(StepArgs& a, const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x,
                     int32_t x_dtype, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, float* x_hat, float* mu,
                     float* log_sigma, void* workspace, int64_t workspace_bytes, void* stream) {
  a = StepArgs{desc, params, static_cast<const bf16*>(shadow_bf16), grads, nullptr, nullptr, eps, seed, offset, row0, rows, 0.f, 0.f,
               0, 0, 0, x_hat, mu, log_sigma, nullptr, workspace, workspace_bytes, static_cast<cudaStream_t>(stream)};
  if (x_dtype == PSVAE_X_F32) a.x = static_cast<const float*>(x);
  else if (x_dtype == PSVAE_X_BF16) a.x16 = static_cast<const bf16*>(x);
  else { set_error("unknown x_dtype %d", x_dtype); return -2; }
  return 0;
}

// The train step behind every psvae_train_fwd_bwd* entry point (psvae_train_fwd_bwd_scoped's arguments; cons == NULL: no consistency term,
// counters == NULL: the host Philox offset).  accumulate (with compute_grads): the step writes this micro-batch's gradient into grad_scratch
// exactly as the non-accumulating step writes `grads`; one pass then adds it (the classifier scope: over the classifier span only -- vae_numel
// is a multiple of 8 floats, so the span stays 16-byte aligned).
static int train_step(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x, int32_t x_dtype,
                      const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, float kl_weight, float clf_weight,
                      int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat, float* mu, float* log_sigma, float* losses,
                      void* workspace, int64_t workspace_bytes, void* stream, const psvae_consistency_desc* cons, const float* cons_params,
                      const int64_t* cons_y, float cons_weight, const psvae_step_counters* counters, int32_t accumulate, float* grad_scratch,
                      int32_t grad_scope) {
  PSVAE_TRY(check_desc(desc, precision));
  const bool acc = accumulate && compute_grads;
  if (acc) {
    if (!grads || !grad_scratch) { set_error("grads and grad_scratch must not be NULL when accumulate != 0"); return -1; }
    if (((reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(grad_scratch)) & 15) != 0) {
      set_error("grads and grad_scratch must be 16-byte aligned");
      return -2;
    }
    if (grads == grad_scratch) { set_error("grad_scratch must not be the gradient buffer"); return -2; }
  }
  StepArgs a;
  PSVAE_TRY(make_step(a, desc, params, shadow_bf16, acc ? grad_scratch : grads, x, x_dtype, eps, seed, offset, row0, rows, x_hat, mu, log_sigma,
                      workspace, workspace_bytes, stream));
  a.y = y; a.kl_w = kl_weight; a.clf_w = clf_weight; a.use_cos = use_cos_loss ? 1 : 0;
  a.want_loss = 1; a.want_grads = compute_grads ? 1 : 0; a.losses = losses;
  a.cons = cons; a.cons_params = cons_params; a.cons_y = cons_y; a.cons_w = cons_weight;
  a.offset_dev = counters ? &counters->rng_offset : nullptr;
  a.grad_scope = grad_scope;
  PSVAE_TRY(precision == PSVAE_BF16 ? run_step<bf16>(a) : run_step<float>(a));
  if (!acc) return 0;
  const int64_t a0 = grad_scope == PSVAE_GRAD_CLASSIFIER ? desc->vae_numel : 0;
  const int64_t n = desc->total_numel - a0;
  launch_dep(grad_accumulate_kernel, dim3(ew_grid(n / 4 + 1)), dim3(256), 0, static_cast<cudaStream_t>(stream), grads + a0,
             (const float*)grad_scratch + a0, n);
  count_launch();
  PSVAE_LAUNCH_CHECK("grad_accumulate_kernel");
  return 0;
}

int psvae_train_fwd_bwd(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x, int32_t x_dtype, const int64_t* y,
                        const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, float kl_weight, float clf_weight,
                        int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat, float* mu, float* log_sigma, float* losses,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  return train_step(desc, params, shadow_bf16, grads, x, x_dtype, y, eps, seed, offset, row0, rows, kl_weight, clf_weight, use_cos_loss, compute_grads,
                    precision, x_hat, mu, log_sigma, losses, workspace, workspace_bytes, stream, nullptr, nullptr, nullptr, 0.f, nullptr, 0, nullptr,
                    PSVAE_GRAD_ALL);
}

int psvae_consistency_desc_init(psvae_consistency_desc* cons, int32_t input_dim, int32_t hidden_dim, int32_t num_classes) {
  if (!cons) { set_error("consistency desc is NULL"); return -1; }
  memset(cons, 0, sizeof(*cons));
  cons->input_dim = input_dim; cons->hidden_dim = hidden_dim; cons->num_classes = num_classes;
  PSVAE_TRY(check_cons(cons));
  const int64_t outs[3] = {hidden_dim, hidden_dim, num_classes}, ins[3] = {input_dim, hidden_dim, hidden_dim};
  int64_t off = 0;
  for (int j = 0; j < 3; ++j) {      // 16-byte aligned blocks (the fp32 engine reads float4)
    cons->w[j] = off; off = align_up64(off + outs[j] * ins[j], 4);
    cons->b[j] = off; off = align_up64(off + outs[j], 4);
  }
  cons->total_numel = align_up64(off, 64);
  return 0;
}

int64_t psvae_consistency_workspace_bytes(const psvae_consistency_desc* cons, int64_t rows, int32_t mode) {
  if (check_cons(cons) != 0) return -1;
  if (rows <= 0 || (mode != PSVAE_MODE_TRAIN && mode != PSVAE_MODE_FORWARD)) { set_error("bad rows/mode"); return -1; }
  Bump b(nullptr);
  ConsBufs w;
  plan_cons(cons, rows, mode == PSVAE_MODE_TRAIN, b, w);
  return b.used + 256;
}

int psvae_consistency_forward(const psvae_consistency_desc* cons, const float* cons_params, const float* x, int64_t rows, float* logits,
                              void* workspace, int64_t workspace_bytes, void* stream) {
  PSVAE_TRY(tc_device_check());
  PSVAE_TRY(check_cons(cons));
  if (rows <= 0) { set_error("rows=%lld must be positive", (long long)rows); return -2; }
  if (!cons_params || !x || !logits) { set_error("cons_params, x and logits must not be NULL"); return -1; }
  ConsBufs w;
  {
    Bump sz(nullptr);
    ConsBufs tmp;
    plan_cons(cons, rows, false, sz, tmp);
    if (sz.used > workspace_bytes || !workspace) {
      set_error("workspace too small: need %lld bytes, got %lld", (long long)sz.used, (long long)workspace_bytes);
      return -2;
    }
    Bump b(workspace);
    plan_cons(cons, rows, false, b, w);
  }
  return cons_forward(cons, cons_params, x, rows, w, logits, static_cast<cudaStream_t>(stream));
}

// scratch of the stand-alone EmbeddingClassifier step on top of the forward / input-gradient chain (plan_cons): split-K and bias partials
struct EmbClfBufs {
  float *wpart = nullptr, *cpart = nullptr;
};
static void plan_embclf(const psvae_consistency_desc* c, int64_t rows, Bump& b, EmbClfBufs& w) {
  int64_t wmax = 0;
  const int64_t outs[3] = {c->hidden_dim, c->hidden_dim, c->num_classes}, ins[3] = {c->input_dim, c->hidden_dim, c->hidden_dim};
  for (int j = 0; j < 3; ++j) {
    const int64_t sp = Engine<float>::wgrad_splits(outs[j], ins[j], rows);
    if (sp * outs[j] * ins[j] > wmax) wmax = sp * outs[j] * ins[j];
  }
  w.wpart = b.take<float>(wmax);
  const int64_t cmax = c->hidden_dim > c->num_classes ? c->hidden_dim : c->num_classes;
  w.cpart = b.take<float>(ceil_div64(rows, g_opt.colsum_rows) * cmax);
}

int64_t psvae_embedding_classifier_workspace_bytes(const psvae_consistency_desc* cons, int64_t rows) {
  if (check_cons(cons) != 0) return -1;
  if (rows <= 0) { set_error("bad rows"); return -1; }
  Bump b(nullptr);
  ConsBufs w;
  EmbClfBufs e;
  plan_cons(cons, rows, true, b, w);
  plan_embclf(cons, rows, b, e);
  return b.used + 256;
}

int psvae_embedding_classifier_step(const psvae_consistency_desc* cons, const float* params, float* grads, const float* x, const int64_t* y, int64_t rows,
                                    int32_t compute_grads, float* logits_out, float* losses, void* workspace, int64_t workspace_bytes, void* stream) {
  PSVAE_TRY(tc_device_check());
  PSVAE_TRY(check_cons(cons));
  if (rows <= 0) { set_error("rows=%lld must be positive", (long long)rows); return -2; }
  if (!params || !x || !y || !losses) { set_error("params, x, y and losses must not be NULL"); return -1; }
  if (compute_grads && !grads) { set_error("grads must not be NULL when compute_grads != 0"); return -1; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ConsBufs w;
  EmbClfBufs e;
  {
    Bump sz(nullptr);
    ConsBufs t1;
    EmbClfBufs t2;
    plan_cons(cons, rows, true, sz, t1);
    plan_embclf(cons, rows, sz, t2);
    if (sz.used > workspace_bytes || !workspace) {
      set_error("workspace too small: need %lld bytes, got %lld", (long long)sz.used, (long long)workspace_bytes);
      return -2;
    }
    Bump b(workspace);
    plan_cons(cons, rows, true, b, w);
    plan_embclf(cons, rows, b, e);
  }
  const int Dm = cons->input_dim, Hm = cons->hidden_dim, C = cons->num_classes;
  PSVAE_TRY(cons_forward(cons, params, x, rows, w, w.logits, st));
  if (logits_out) PSVAE_CUDA(cudaMemcpyAsync(logits_out, w.logits, (size_t)rows * C * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // CrossEntropyLoss (mean) + multiclass accuracy; logits become d loss / d logits in place
  launch_dep(ce_kernel, dim3((unsigned)w.n_ce), dim3(256), 0, st, w.logits, y, rows, C, 1.f / (float)rows, compute_grads ? 1 : 0, w.nll_part, w.acc_part);
  count_launch();
  PSVAE_LAUNCH_CHECK("ce_kernel");
  LossPartials lp;
  memset(&lp, 0, sizeof(lp));
  lp.inv_b = 1.f / (float)rows;
  lp.cons_nll = w.nll_part; lp.cons_acc = w.acc_part; lp.n_cons = (int)w.n_ce; lp.cons_w = 1.f;
  launch_dep(finalize_losses_kernel, dim3(1), dim3(1024), 0, st, lp, losses);      // losses[0] = losses[12] = CE, losses[13] = accuracy
  count_launch();
  PSVAE_LAUNCH_CHECK("finalize_losses_kernel");
  if (!compute_grads) return 0;
  PSVAE_CUDA(cudaMemsetAsync(grads, 0, (size_t)cons->total_numel * sizeof(float), st));
  StepBufs<float> sb;
  sb.wpart = e.wpart; sb.cpart = e.cpart;
  // fc3, then back through the two ReLU layers (embedding_classifier.py:50-62 under autograd)
  PSVAE_TRY(wgrad_clf<float>(w.logits, C, w.a2, Hm, rows, C, Hm, grads + cons->w[2], grads + cons->b[2], sb, st));
  PSVAE_TRY(clf_dgrad(ACT_RELU, w.logits, C, params + cons->w[2], Hm, w.a2, w.g2, 0.f, rows, st));
  PSVAE_TRY(wgrad_clf<float>(w.g2, Hm, w.a1, Hm, rows, Hm, Hm, grads + cons->w[1], grads + cons->b[1], sb, st));
  PSVAE_TRY(clf_dgrad(ACT_RELU, w.g2, Hm, params + cons->w[1], Hm, w.a1, w.g1, 0.f, rows, st));
  PSVAE_TRY(wgrad_clf<float>(w.g1, Hm, x, Dm, rows, Hm, Dm, grads + cons->w[0], grads + cons->b[0], sb, st));
  return 0;
}

int psvae_train_fwd_bwd_consistency(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x, int32_t x_dtype,
                                    const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, float kl_weight,
                                    float clf_weight, int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat, float* mu,
                                    float* log_sigma, float* losses, void* workspace, int64_t workspace_bytes, void* stream,
                                    const psvae_consistency_desc* cons, const float* cons_params, const int64_t* cons_y, float cons_weight) {
  PSVAE_TRY(check_desc(desc, precision));
  if (!cons) { set_error("consistency desc is NULL (use psvae_train_fwd_bwd for a step without the consistency term)"); return -1; }
  return train_step(desc, params, shadow_bf16, grads, x, x_dtype, y, eps, seed, offset, row0, rows, kl_weight, clf_weight, use_cos_loss, compute_grads,
                    precision, x_hat, mu, log_sigma, losses, workspace, workspace_bytes, stream, cons, cons_params, cons_y, cons_weight, nullptr, 0,
                    nullptr, PSVAE_GRAD_ALL);
}

int psvae_train_fwd_bwd_dc(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x, int32_t x_dtype,
                           const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, float kl_weight, float clf_weight,
                           int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat, float* mu, float* log_sigma, float* losses,
                           void* workspace, int64_t workspace_bytes, void* stream, const psvae_consistency_desc* cons, const float* cons_params,
                           const int64_t* cons_y, float cons_weight, const psvae_step_counters* counters) {
  return train_step(desc, params, shadow_bf16, grads, x, x_dtype, y, eps, seed, offset, row0, rows, kl_weight, clf_weight, use_cos_loss, compute_grads,
                    precision, x_hat, mu, log_sigma, losses, workspace, workspace_bytes, stream, cons, cons_params, cons_y, cons_weight, counters, 0,
                    nullptr, PSVAE_GRAD_ALL);
}

int psvae_train_fwd_bwd_acc(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x, int32_t x_dtype,
                            const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, float kl_weight, float clf_weight,
                            int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat, float* mu, float* log_sigma, float* losses,
                            void* workspace, int64_t workspace_bytes, void* stream, const psvae_consistency_desc* cons, const float* cons_params,
                            const int64_t* cons_y, float cons_weight, const psvae_step_counters* counters, int32_t accumulate, float* grad_scratch) {
  return train_step(desc, params, shadow_bf16, grads, x, x_dtype, y, eps, seed, offset, row0, rows, kl_weight, clf_weight, use_cos_loss, compute_grads,
                    precision, x_hat, mu, log_sigma, losses, workspace, workspace_bytes, stream, cons, cons_params, cons_y, cons_weight, counters,
                    accumulate, grad_scratch, PSVAE_GRAD_ALL);
}

int psvae_train_fwd_bwd_scoped(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x,
                               int32_t x_dtype, const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows,
                               float kl_weight, float clf_weight, int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat,
                               float* mu, float* log_sigma, float* losses, void* workspace, int64_t workspace_bytes, void* stream,
                               const psvae_consistency_desc* cons, const float* cons_params, const int64_t* cons_y, float cons_weight,
                               const psvae_step_counters* counters, int32_t accumulate, float* grad_scratch, int32_t grad_scope) {
  // argument checks first: they do not need a device
  PSVAE_TRY(check_desc(desc, precision));
  if (grad_scope != PSVAE_GRAD_ALL && grad_scope != PSVAE_GRAD_CLASSIFIER) { set_error("unknown grad_scope %d", grad_scope); return -2; }
  if (grad_scope == PSVAE_GRAD_CLASSIFIER && desc->clf_num_heads <= 0) {
    set_error("grad_scope PSVAE_GRAD_CLASSIFIER: the model has no latent classifier");
    return -2;
  }
  return train_step(desc, params, shadow_bf16, grads, x, x_dtype, y, eps, seed, offset, row0, rows, kl_weight, clf_weight, use_cos_loss, compute_grads,
                    precision, x_hat, mu, log_sigma, losses, workspace, workspace_bytes, stream, cons, cons_params, cons_y, cons_weight, counters,
                    accumulate, grad_scratch, grad_scope);
}

int psvae_vae_backward(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x, int32_t x_dtype, const float* eps,
                       uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, int32_t precision, const float* g_x_hat, const float* g_mu,
                       const float* g_log_sigma, void* workspace, int64_t workspace_bytes, void* stream) {
  PSVAE_TRY(check_desc(desc, precision));
  StepArgs a;
  PSVAE_TRY(make_step(a, desc, params, shadow_bf16, grads, x, x_dtype, eps, seed, offset, row0, rows, nullptr, nullptr, nullptr, workspace,
                      workspace_bytes, stream));
  a.want_grads = 1;
  a.ext = 1; a.ext_gx = g_x_hat; a.ext_gmu = g_mu; a.ext_gls = g_log_sigma;
  return precision == PSVAE_BF16 ? run_step<bf16>(a) : run_step<float>(a);
}

int psvae_forward(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, const void* x, int32_t x_dtype, const float* eps, uint64_t seed,
                  uint64_t offset, int64_t row0, int64_t rows, int32_t precision, float* x_hat, float* mu, float* log_sigma, void* workspace,
                  int64_t workspace_bytes, void* stream) {
  PSVAE_TRY(check_desc(desc, precision));
  if (!x_hat) { set_error("x_hat must not be NULL"); return -1; }
  StepArgs a;
  PSVAE_TRY(make_step(a, desc, params, shadow_bf16, nullptr, x, x_dtype, eps, seed, offset, row0, rows, x_hat, mu, log_sigma, workspace,
                      workspace_bytes, stream));
  return precision == PSVAE_BF16 ? run_step<bf16>(a) : run_step<float>(a);
}

int psvae_decode(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, const float* z, uint64_t seed, uint64_t offset,
                 int64_t row0, int64_t rows, int32_t precision, float* x_hat, float* z_out, void* workspace, int64_t workspace_bytes, void* stream) {
  PSVAE_TRY(check_desc(desc, precision));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return precision == PSVAE_BF16
             ? run_decode<bf16>(desc, params, static_cast<const bf16*>(shadow_bf16), z, seed, offset, row0, rows, x_hat, z_out, workspace, workspace_bytes, st)
             : run_decode<float>(desc, params, nullptr, z, seed, offset, row0, rows, x_hat, z_out, workspace, workspace_bytes, st);
}

}  // extern "C"

// The classifier part of LangevinClf (everything but the targets) from the model description.
static LangevinClf langevin_clf(const psvae_model_desc* desc) {
  Net n(desc);
  LangevinClf c;
  memset(&c, 0, sizeof(c));
  c.L = n.L; c.n_trunk = desc->clf_num_trunk; c.hidden = desc->clf_num_trunk ? desc->clf_hidden : 0;
  c.act = desc->clf_activation; c.n_heads = desc->clf_num_heads;
  int off = 0;
  for (int t = 0; t < c.n_trunk; ++t) {
    c.g_trunk_w[t] = desc->clf_trunk_w[t]; c.g_trunk_b[t] = desc->clf_trunk_b[t];
    c.s_trunk_w[t] = off; off += desc->clf_hidden * n.clf_trunk_in(t);
    c.s_trunk_b[t] = off; off += desc->clf_hidden;
  }
  for (int h = 0; h < c.n_heads; ++h) {
    c.head_classes[h] = desc->clf_head_classes[h];
    c.g_head_w[h] = desc->clf_head_w[h]; c.g_head_b[h] = desc->clf_head_b[h];
    c.s_head_w[h] = off; off += c.head_classes[h] * n.clf_feat();
    c.s_head_b[h] = off; off += c.head_classes[h];
  }
  for (int h = 0; h < 4; ++h) c.targets[h] = -1;
  c.w_floats = off;
  return c;
}

// Launch the Langevin loop: the shared-target instances for rt == NULL, the per-row ones otherwise.  c.targets[h] >= 0 marks the heads the
// kernel stages (and, for the shared instances, their targets).
template <bool ROW_TARGETS>
static int langevin_launch(const LangevinClf& c, const LangevinRows& rt, const float* params, float* z_io, int64_t rows, float step_size,
                           int32_t num_steps, float noise_weight, uint64_t seed, uint64_t offset0, int64_t row0, int32_t init_from_philox,
                           const float* noise, float* history, float* stats, float prior_weight, float threshold, int32_t* stop_step,
                           float* last_prob, cudaStream_t st) {
  if (stats && num_steps > 0) PSVAE_CUDA(cudaMemsetAsync(stats, 0, sizeof(float) * 2 * (size_t)num_steps, st));
  // fast path: linear heads on z, one thread per sample (langevin_fast_kernel)
  int targeted_classes = 0;
  for (int h = 0; h < c.n_heads; ++h)
    if (c.targets[h] >= 0) targeted_classes += c.head_classes[h];
  if (c.n_trunk == 0 && targeted_classes <= CLF_LG_MAXC && (c.L == 16 || c.L == 32 || c.L == 64) && !g_opt.langevin_generic) {
    const unsigned gridf = (unsigned)ceil_div64(rows, LGF_THREADS);
    switch (c.L) {
      case 16: launch_dep(langevin_fast_kernel<16, ROW_TARGETS>, dim3(gridf), dim3(LGF_THREADS), 0, st, c, params, z_io, rows, step_size, num_steps, noise_weight, seed, offset0, row0, init_from_philox, noise, history, stats, prior_weight, threshold, stop_step, last_prob, rt); break;
      case 32: launch_dep(langevin_fast_kernel<32, ROW_TARGETS>, dim3(gridf), dim3(LGF_THREADS), 0, st, c, params, z_io, rows, step_size, num_steps, noise_weight, seed, offset0, row0, init_from_philox, noise, history, stats, prior_weight, threshold, stop_step, last_prob, rt); break;
      default: launch_dep(langevin_fast_kernel<64, ROW_TARGETS>, dim3(gridf), dim3(LGF_THREADS), 0, st, c, params, z_io, rows, step_size, num_steps, noise_weight, seed, offset0, row0, init_from_philox, noise, history, stats, prior_weight, threshold, stop_step, last_prob, rt); break;
    }
    count_launch();
    PSVAE_LAUNCH_CHECK("langevin_fast_kernel");
    return 0;
  }
  const size_t smem = langevin_smem_bytes(c, ROW_TARGETS);
  if (smem > 227 * 1024) { set_error("classifier too large for the Langevin kernel's shared memory (%zu bytes)", smem); return -2; }
  PSVAE_CUDA(cudaFuncSetAttribute(langevin_kernel<ROW_TARGETS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)ceil_div64(rows, LG_TILE);
  launch_dep(langevin_kernel<ROW_TARGETS>, dim3(grid), dim3(LG_THREADS), smem, st, c, params, z_io, rows, step_size, num_steps, noise_weight, seed, offset0,
             row0, init_from_philox, noise, history, stats, prior_weight, threshold, stop_step, last_prob, rt);
  count_launch();
  PSVAE_LAUNCH_CHECK("langevin_kernel");
  return 0;
}

extern "C" {

int psvae_langevin(const psvae_model_desc* desc, const float* params, float* z_io, int64_t rows, const int32_t* targets_host, float step_size,
                   int32_t num_steps, float noise_weight, uint64_t seed, uint64_t offset0, int64_t row0, int32_t init_from_philox,
                   const float* noise, float* history, float* stats, float prior_weight, float threshold, int32_t* stop_step, float* last_prob,
                   void* stream) {
  PSVAE_TRY(check_desc(desc, PSVAE_FP32));
  PSVAE_TRY(tc_device_check());
  if (!params || !z_io || !targets_host) { set_error("params, z_io, targets must not be NULL"); return -1; }
  if (desc->clf_num_heads <= 0) { set_error("conditional synthesis needs a latent classifier (ps_vae/inference.py:80)"); return -2; }
  if (rows <= 0) { set_error("rows must be positive"); return -2; }
  if (num_steps < 0) { set_error("num_steps must be >= 0"); return -2; }
  LangevinClf c = langevin_clf(desc);
  int any = 0;
  for (int h = 0; h < c.n_heads; ++h) {
    c.targets[h] = targets_host[h];
    if (c.targets[h] >= c.head_classes[h]) { set_error("target %d of head %d is out of range (%d classes)", c.targets[h], h, c.head_classes[h]); return -2; }
    if (c.targets[h] >= 0) any = 1;
  }
  if (!any) { set_error("classifier_target selects no head"); return -2; }
  LangevinRows rt;
  memset(&rt, 0, sizeof(rt));
  return langevin_launch<false>(c, rt, params, z_io, rows, step_size, num_steps, noise_weight, seed, offset0, row0, init_from_philox, noise, history,
                                stats, prior_weight, threshold, stop_step, last_prob, static_cast<cudaStream_t>(stream));
}

int psvae_langevin_rows(const psvae_model_desc* desc, const float* params, float* z_io, int64_t rows, const int32_t* row_targets, int32_t n_mix,
                        const int32_t* mix_targets_host, const uint32_t* mix_thresholds_host, int32_t* row_targets_out, float step_size,
                        int32_t num_steps, float noise_weight, uint64_t seed, uint64_t offset0, int64_t row0, int32_t init_from_philox,
                        const float* noise, float* history, float* stats, float prior_weight, float threshold, int32_t* stop_step, float* last_prob,
                        void* stream) {
  static_assert(PSVAE_MAX_TARGET_MIX == LG_MAX_MIX, "target mix capacity");
  // argument checks first: they do not need a device
  PSVAE_TRY(check_desc(desc, PSVAE_FP32));
  if (desc->clf_num_heads <= 0) { set_error("conditional synthesis needs a latent classifier (ps_vae/inference.py:80)"); return -2; }
  if (n_mix < 0 || n_mix > PSVAE_MAX_TARGET_MIX) { set_error("n_mix=%d out of range [0,%d]", n_mix, PSVAE_MAX_TARGET_MIX); return -2; }
  if ((row_targets != nullptr) == (n_mix > 0)) { set_error("give exactly one of row_targets and a target mix (n_mix >= 1)"); return -2; }
  LangevinClf c = langevin_clf(desc);
  LangevinRows rt;
  memset(&rt, 0, sizeof(rt));
  rt.targets = row_targets;
  if (row_targets) {
    for (int h = 0; h < c.n_heads; ++h) c.targets[h] = 0;         // any head can be named by some row
  } else {
    if (!mix_targets_host || (n_mix > 1 && !mix_thresholds_host)) { set_error("a target mix needs its targets and n_mix - 1 thresholds"); return -1; }
    if (!row_targets_out) { set_error("a target mix needs row_targets_out for the drawn targets"); return -1; }
    rt.targets_out = row_targets_out;
    rt.n_mix = n_mix;
    rt.mix_offset = offset0 + (uint64_t)num_steps + 1;
    for (int k = 0; k < n_mix; ++k) {
      uint32_t p = 0;
      for (int h = 0; h < PSVAE_MAX_CLF_HEADS; ++h) {
        const int t = mix_targets_host[k * PSVAE_MAX_CLF_HEADS + h];
        if (t == -1) continue;
        if (h >= c.n_heads || t < 0 || t >= c.head_classes[h]) { set_error("mix entry %d: target %d of head %d is out of range", k, t, h); return -2; }
        p |= (uint32_t)(t + 1) << (8 * h);
        c.targets[h] = 0;
      }
      if (!p) { set_error("mix entry %d names no head", k); return -2; }
      rt.mix[k] = p;
    }
    for (int k = 0; k + 1 < n_mix; ++k) {
      rt.thr[k] = mix_thresholds_host[k];
      if (k > 0 && rt.thr[k] < rt.thr[k - 1]) { set_error("mix thresholds must not decrease (entry %d)", k); return -2; }
    }
  }
  PSVAE_TRY(tc_device_check());
  if (!params || !z_io) { set_error("params, z_io must not be NULL"); return -1; }
  if (rows <= 0) { set_error("rows must be positive"); return -2; }
  if (num_steps < 0) { set_error("num_steps must be >= 0"); return -2; }
  return langevin_launch<true>(c, rt, params, z_io, rows, step_size, num_steps, noise_weight, seed, offset0, row0, init_from_philox, noise, history,
                               stats, prior_weight, threshold, stop_step, last_prob, static_cast<cudaStream_t>(stream));
}

int psvae_gemm_bf16(const void* a_bf16, const void* b_bf16, const float* bias, float* c, int64_t m, int32_t n, int64_t k, int32_t a_mn, int32_t b_mn,
                    int32_t relu, int32_t split_k, void* workspace, int64_t workspace_bytes, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!a_bf16 || !b_bf16 || !c) { set_error("a, b, c must not be NULL"); return -1; }
  if (m <= 0 || n <= 0 || k <= 0) { set_error("m, n, k must be positive"); return -2; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bf16* A = static_cast<const bf16*>(a_bf16);
  const bf16* B = static_cast<const bf16*>(b_bf16);
  TcOperand oa{A, m, a_mn ? m : k, a_mn != 0};
  TcOperand ob{B, (int64_t)n, b_mn ? (int64_t)n : k, b_mn != 0};
  const int fbn = (int)g_opt.tc_force_bn;
  if (split_k > 1) {
    const int64_t kb = ceil_div64(k, TC_BK);
    int64_t s = split_k > kb ? kb : split_k;
    const int64_t per = ceil_div64(kb, s);
    s = ceil_div64(kb, per);
    if (!workspace || workspace_bytes < (int64_t)(s * m * n * (int64_t)sizeof(float))) {
      set_error("split-K needs %lld bytes of workspace", (long long)(s * m * n * (int64_t)sizeof(float)));
      return -2;
    }
    float* part = static_cast<float*>(workspace);
    EpiStore e{part, n, m * n, 1.f, 0.f, nullptr, 0};
    int r;
    if (a_mn && b_mn) r = gemm_tc_launch<true, true>(oa, ob, m, n, k, (int)s, e, st, fbn);
    else if (!a_mn && b_mn) r = gemm_tc_launch<false, true>(oa, ob, m, n, k, (int)s, e, st, fbn);
    else if (!a_mn && !b_mn) r = gemm_tc_launch<false, false>(oa, ob, m, n, k, (int)s, e, st, fbn);
    else { set_error("a_mn && !b_mn is not used by this library"); return -2; }
    PSVAE_TRY(r);
    return launch_reduce(part, m * n, (int)s, c, st);
  }
  if (a_mn && b_mn) {
    EpiStore e{c, n, 0, 1.f, 0.f, nullptr, 0};
    return gemm_tc_launch<true, true>(oa, ob, m, n, k, 1, e, st, fbn);
  }
  if (a_mn) { set_error("a_mn && !b_mn is not used by this library"); return -2; }
  if (b_mn) {
    if (relu || bias) { set_error("bias/relu are only wired for the K-major x K-major form"); return -2; }
    EpiStore e{c, n, 0, 1.f, 0.f, nullptr, 0};
    return gemm_tc_launch<false, true>(oa, ob, m, n, k, 1, e, st, fbn);
  }
  if (relu) {
    EpiBiasAct<float, ACT_RELU> e{bias, c, n, nullptr};
    return gemm_tc_launch<false, false>(oa, ob, m, n, k, 1, e, st, fbn);
  }
  EpiBiasAct<float, ACT_NONE> e{bias, c, n, nullptr};
  return gemm_tc_launch<false, false>(oa, ob, m, n, k, 1, e, st, fbn);
}

// Profiling probe: the two hot epilogue forms of the train step on free-standing operands.
//   form 0: out = relu(A W^T + bias) in bf16 (+ ReLU bit mask when mask != NULL)          (forward Linear, model.py:14-36)
//   form 1: out = (A W) .* mask in bf16 (+ column sums into colsum when colsum != NULL)   (dgrad through a hidden Linear)
// out == NULL skips the store (mainloop + TMEM read only).
int psvae_gemm_probe(const void* a_bf16, const void* w_bf16, const float* bias, void* out_bf16, uint32_t* mask, float* colsum, int64_t m, int32_t n,
                     int64_t k, int32_t form, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!a_bf16 || !w_bf16) { set_error("a, w must not be NULL"); return -1; }
  if (m <= 0 || n <= 0 || k <= 0) { set_error("m, n, k must be positive"); return -2; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bf16* A = static_cast<const bf16*>(a_bf16);
  const bf16* W = static_cast<const bf16*>(w_bf16);
  bf16* out = static_cast<bf16*>(out_bf16);
  const int fbn = (int)g_opt.tc_force_bn;
  if (form == 0) {
    TcOperand oa{A, m, k, false};
    TcOperand ob{W, (int64_t)n, k, false};          // W [n][k]
    EpiBiasAct<bf16, ACT_RELU> e{bias, out, n, nullptr, mask, m};
    return gemm_tc_launch<false, false>(oa, ob, m, n, k, 1, e, st, fbn);
  }
  if (form == 1) {
    if (!mask) { set_error("form 1 needs a mask"); return -1; }
    TcOperand oa{A, m, k, false};
    TcOperand ob{W, (int64_t)n, (int64_t)n, true};  // W [k][n] as stored (out = k, in = n)
    if (colsum) {
      EpiActGrad<bf16, bf16, ACT_RELU, true> e{nullptr, 0, mask, m, out, n, 0.f, nullptr, colsum, 1};
      return gemm_tc_launch<false, true>(oa, ob, m, n, k, 1, e, st, fbn);
    }
    EpiActGrad<bf16, bf16, ACT_RELU, false> e{nullptr, 0, mask, m, out, n, 0.f, nullptr, nullptr, 0};
    return gemm_tc_launch<false, true>(oa, ob, m, n, k, 1, e, st, fbn);
  }
  if (form == 2) {      // wgrad: out[n_out = n][n_in = k] (fp32, accumulated by TMA reduce-add) = A[m][n]^T * W[m][k]   (m = batch rows)
    float* gw = static_cast<float*>(out_bf16);
    if (!gw) { set_error("form 2 needs an output"); return -1; }
    const int out_dim = n, in_dim = (int)k;
    const int splits = Engine<bf16>::wgrad_splits(out_dim, in_dim, m);
    EpiStore e{gw, in_dim, 0, 1.f, 0.f, nullptr, 1};
    return Engine<bf16>::gemm<G_WGRAD>(A, out_dim, W, in_dim, out_dim, in_dim, m, splits, true, e, st);
  }
  set_error("unknown probe form %d", form);
  return -2;
}

int psvae_gemm_fp32(const float* a, const float* b, const float* bias, float* c, int64_t m, int32_t n, int64_t k, int32_t a_mn, int32_t b_mn,
                    int32_t relu, void* stream) {
  PSVAE_TRY(tc_device_check());
  if (!a || !b || !c) { set_error("a, b, c must not be NULL"); return -1; }
  if (m <= 0 || n <= 0 || k <= 0) { set_error("m, n, k must be positive"); return -2; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SgemmOperand oa{a, a_mn ? 1 : k, a_mn ? m : 1};
  SgemmOperand ob{b, b_mn ? 1 : k, b_mn ? (int64_t)n : 1};
  const bool vec = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(c) & 15) == 0) && (!bias || (reinterpret_cast<uintptr_t>(bias) & 15) == 0);
  if (relu) {
    EpiBiasAct<float, ACT_RELU> e{bias, c, n, nullptr};
    return sgemm_launch(oa, ob, m, n, k, 1, vec, e, st);
  }
  EpiBiasAct<float, ACT_NONE> e{bias, c, n, nullptr};
  return sgemm_launch(oa, ob, m, n, k, 1, vec, e, st);
}

}  // extern "C"

// =================================================================================================
// cosine top-k search (cosine_topk.cuh)
// =================================================================================================
namespace psvae {

// Workspace carving and work split of one psvae_cosine_topk call.  Depends on the arguments and the option "topk_key_splits" only (not on the
// device), so psvae_cosine_topk_workspace_bytes answers without a GPU.
struct TopkPlan {
  int64_t m_tiles, k_tiles, splits, tiles_per_split;
  int64_t off_qn, off_kn, off_iq, off_ik, off_part, bytes;
};

static int topk_plan(int64_t nq, int64_t nk, int32_t dim, int32_t k, TopkPlan* p) {
  if (nq <= 0 || nk <= 0) { set_error("nq and nk must be positive (nq=%lld nk=%lld)", (long long)nq, (long long)nk); return -2; }
  if (nq > INT32_MAX || nk > INT32_MAX) { set_error("nq and nk must be < 2^31 (tensor-map coordinates)"); return -2; }
  if (dim <= 0 || dim % 8 != 0 || dim > TK_MAX_DIM) { set_error("dim=%d: must be a positive multiple of 8, at most %d", dim, TK_MAX_DIM); return -2; }
  if (k < 1 || k > TK_MAX_K) { set_error("k=%d out of range [1,%d]", k, TK_MAX_K); return -2; }
  p->m_tiles = ceil_div64(nq, TK_BM);
  p->k_tiles = ceil_div64(nk, TK_BN);
  int64_t s = g_opt.topk_key_splits;
  if (s <= 0) {
    // few query tiles: split the key range so that (query tile, key range) items fill whole rounds of the persistent grid -- the
    // fewest splits within 2 % of the best round efficiency among those giving at least one item per SM
    s = 1;
    if (p->m_tiles < 4 * PSVAE_NUM_SMS) {
      const int64_t lo = std::min<int64_t>(p->k_tiles, ceil_div64(PSVAE_NUM_SMS, p->m_tiles)), hi = std::min<int64_t>(p->k_tiles, 4 * lo);
      double best = -1.0;
      for (int64_t c = lo; c <= hi; ++c) {
        const int64_t items = p->m_tiles * ceil_div64(p->k_tiles, ceil_div64(p->k_tiles, c));
        const double eff = (double)items / (double)(ceil_div64(items, PSVAE_NUM_SMS) * PSVAE_NUM_SMS);
        if (eff > best + 0.02) { best = eff; s = c; }
      }
    }
  }
  if (s > p->k_tiles) s = p->k_tiles;
  p->tiles_per_split = ceil_div64(p->k_tiles, s);
  p->splits = ceil_div64(p->k_tiles, p->tiles_per_split);     // no empty key range
  const int64_t C = 2 * (int64_t)k;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { const int64_t o = off; off = align_up64(off + bytes, 256); return o; };
  p->off_qn = take(nq * dim * 2);
  p->off_kn = take(nk * dim * 2);
  p->off_iq = take(nq * 4);
  p->off_ik = take(nk * 4);
  p->off_part = take(p->splits * p->m_tiles * TK_BM * C * 8);
  p->bytes = off;
  return 0;
}

template <typename TQ, typename TK, bool LARGEST>
static int topk_launch(const TopkPlan& p, const void* q, int64_t nq, int64_t q_row0, const void* keys, int64_t nk, int64_t k_row0, int32_t dim,
                       int32_t k, bool excl, float* out_sim, int64_t* out_idx, uint8_t* ws, cudaStream_t st) {
  const TQ* qt = static_cast<const TQ*>(q);
  const TK* kt = static_cast<const TK*>(keys);
  bf16* qn = reinterpret_cast<bf16*>(ws + p.off_qn);
  bf16* kn = reinterpret_cast<bf16*>(ws + p.off_kn);
  float* iq = reinterpret_cast<float*>(ws + p.off_iq);
  float* ik = reinterpret_cast<float*>(ws + p.off_ik);
  int2* part = reinterpret_cast<int2*>(ws + p.off_part);
  const int C = 2 * k;

  topk_normalize_kernel<TQ><<<ew_grid(nq * 32), 256, 0, st>>>(qt, nq, dim, qn, iq);
  count_launch();
  PSVAE_LAUNCH_CHECK("topk_normalize_kernel");
  topk_normalize_kernel<TK><<<ew_grid(nk * 32), 256, 0, st>>>(kt, nk, dim, kn, ik);
  count_launch();
  PSVAE_LAUNCH_CHECK("topk_normalize_kernel");

  CUtensorMap tq, tk;
  PSVAE_TRY(tc_tensor_map(TcOperand{qn, nq, dim, false}, dim, TK_BM, &tq));
  PSVAE_TRY(tc_tensor_map(TcOperand{kn, nk, dim, false}, dim, TK_BN, &tk));
  TopkShape s;
  memset(&s, 0, sizeof(s));
  s.nk = nk;
  s.q_row0 = q_row0;
  s.k_row0 = k_row0;
  s.kb = (int32_t)ceil_div64(dim, TK_BK);
  s.C = C;
  s.m_tiles = (int32_t)p.m_tiles;
  s.k_tiles = (int32_t)p.k_tiles;
  s.splits = (int32_t)p.splits;
  s.tiles_per_split = (int32_t)p.tiles_per_split;
  s.exclude_self = excl ? 1 : 0;
  s.part = part;
  // shared memory: [barriers 1 KB][candidate lists C x 128 x 8 B][query tile kb x 16 KB][key ring stages x 32 KB]
  s.list_off = TK_BAR_BYTES;
  s.q_off = s.list_off + (uint32_t)align_up64((int64_t)C * TK_BM * 8, 1024);
  s.ring_off = s.q_off + (uint32_t)(s.kb * TK_QBLOCK_BYTES);
  const int64_t room = (int64_t)TK_SMEM_MAX - 1024 /*align slack*/ - s.ring_off;
  s.stages = (int32_t)std::min<int64_t>(TK_MAX_STAGES, room / TK_STAGE_BYTES);
  if (s.stages < 2) { set_error("cosine top-k: no room for the key ring (dim=%d, k=%d)", dim, k); return -2; }
  const size_t smem = (size_t)s.ring_off + (size_t)s.stages * TK_STAGE_BYTES + 1024;
  auto kern = topk_search_kernel<LARGEST>;
  static unsigned long long attr_mask = 0;   // per instantiation, one bit per device
  int dev = 0;
  PSVAE_CUDA(cudaGetDevice(&dev));
  if (!(attr_mask >> (dev & 63) & 1ull)) {
    PSVAE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, TK_SMEM_MAX));
    attr_mask |= 1ull << (dev & 63);
  }
  const int64_t items = p.m_tiles * p.splits;
  const int grid = (int)std::min<int64_t>(items, tc_grid_size());
  kern<<<grid, TK_THREADS, smem, st>>>(tq, tk, s);
  count_launch();
  PSVAE_LAUNCH_CHECK("topk_search_kernel");

  topk_merge_kernel<TQ, TK, LARGEST><<<ew_grid(nq * 32), 256, 0, st>>>(part, p.m_tiles * TK_BM, (int)p.splits, C, k, qt, kt, iq, ik, nq, dim, k_row0,
                                                                  out_sim, out_idx);
  count_launch();
  PSVAE_LAUNCH_CHECK("topk_merge_kernel");
  return 0;
}

template <typename TQ>
static int topk_dispatch(int32_t k_dtype, bool smallest, const TopkPlan& p, const void* q, int64_t nq, int64_t q_row0, const void* keys, int64_t nk,
                         int64_t k_row0, int32_t dim, int32_t k, bool excl, float* out_sim, int64_t* out_idx, uint8_t* ws, cudaStream_t st) {
  if (k_dtype == PSVAE_X_F32) {
    return smallest ? topk_launch<TQ, float, false>(p, q, nq, q_row0, keys, nk, k_row0, dim, k, excl, out_sim, out_idx, ws, st)
                    : topk_launch<TQ, float, true>(p, q, nq, q_row0, keys, nk, k_row0, dim, k, excl, out_sim, out_idx, ws, st);
  }
  return smallest ? topk_launch<TQ, bf16, false>(p, q, nq, q_row0, keys, nk, k_row0, dim, k, excl, out_sim, out_idx, ws, st)
                  : topk_launch<TQ, bf16, true>(p, q, nq, q_row0, keys, nk, k_row0, dim, k, excl, out_sim, out_idx, ws, st);
}

}  // namespace psvae

extern "C" {

int64_t psvae_cosine_topk_workspace_bytes(int64_t nq, int64_t nk, int32_t dim, int32_t k) {
  TopkPlan p;
  if (topk_plan(nq, nk, dim, k, &p) != 0) return -1;
  return p.bytes;
}

int psvae_cosine_topk(const void* q, int32_t q_dtype, int64_t nq, int64_t q_row0, const void* keys, int32_t k_dtype, int64_t nk, int64_t k_row0,
                      int32_t dim, int32_t k, int32_t flags, float* out_sim, int64_t* out_idx, void* workspace, int64_t workspace_bytes, void* stream) {
  // argument checks first: they do not need a device
  if ((q_dtype != PSVAE_X_F32 && q_dtype != PSVAE_X_BF16) || (k_dtype != PSVAE_X_F32 && k_dtype != PSVAE_X_BF16)) {
    set_error("q_dtype=%d k_dtype=%d: each must be PSVAE_X_F32 or PSVAE_X_BF16", q_dtype, k_dtype);
    return -2;
  }
  if (flags & ~(PSVAE_TOPK_SMALLEST | PSVAE_TOPK_EXCLUDE_SELF)) { set_error("unknown flags 0x%x", flags); return -2; }
  if (q_row0 < 0 || k_row0 < 0) { set_error("q_row0 and k_row0 must be >= 0"); return -2; }
  TopkPlan p;
  PSVAE_TRY(topk_plan(nq, nk, dim, k, &p));
  const bool excl = (flags & PSVAE_TOPK_EXCLUDE_SELF) != 0;
  if (k > nk - (excl ? 1 : 0)) { set_error("k=%d exceeds the %lld keys available%s", k, (long long)(nk - (excl ? 1 : 0)), excl ? " (exclude_self)" : ""); return -2; }
  if (workspace_bytes < p.bytes) { set_error("workspace of %lld bytes is too small: need %lld", (long long)workspace_bytes, (long long)p.bytes); return -2; }
  PSVAE_TRY(tc_device_check());
  if (!q || !keys || !out_sim || !out_idx || !workspace) { set_error("q, keys, out_sim, out_idx, workspace must not be NULL"); return -1; }
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) { set_error("workspace must be 256-byte aligned"); return -2; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const bool smallest = (flags & PSVAE_TOPK_SMALLEST) != 0;
  if (q_dtype == PSVAE_X_F32) return topk_dispatch<float>(k_dtype, smallest, p, q, nq, q_row0, keys, nk, k_row0, dim, k, excl, out_sim, out_idx, ws, st);
  return topk_dispatch<bf16>(k_dtype, smallest, p, q, nq, q_row0, keys, nk, k_row0, dim, k, excl, out_sim, out_idx, ws, st);
}

}  // extern "C"
