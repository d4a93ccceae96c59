// libfear_b200.so -- executor + C ABI of the FEAR-XS hot path on B200 (sm_100a).
// See include/fear_b200.h for the contract and DESIGN.md for the data layout.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/fear_b200.h"
#include "arch.h"
#include "kernels_ffma.cuh"
#include "kernels_tc.cuh"
#include "kernels_dw_tma.cuh"
#include "kernels_stem_fused.cuh"
#include "kernels_irf_fused.cuh"
#include "kernels_dwpw_small.cuh"
#include "kernels_multitrack.cuh"

using namespace fear;

// ------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";

static int set_err(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                           \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return set_err((int)_e, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define FEAR_TRY(expr)       \
  do {                       \
    int _r = (expr);         \
    if (_r != 0) return _r;  \
  } while (0)

// ------------------------------------------------------------------------------ stages
enum Stage {
  ST_STEM = 0,
  ST_BACKBONE_PW,
  ST_BACKBONE_DW,
  ST_NECK,
  ST_HEAD_DW,
  ST_HEAD_PW,
  ST_CORR,
  ST_PRED,
  ST_DECODE,
  ST_LAYOUT,
  ST_COUNT
};
static const char* kStageNames[ST_COUNT] = {"stem",    "backbone_pw", "backbone_dw", "neck",   "head_dw",
                                            "head_pw", "corr",        "pred",        "decode", "layout"};

enum Impl { IMPL_FFMA = 0, IMPL_TC = 1 };  // CUDA cores (FFMA baseline / fallback shapes) | tcgen05

struct Options {
  int corr = -1;  // -1 = auto: tcgen05 when the tensor-core path initialised on this device, else CUDA cores
  int pw = -1;
  int fuse_dwpw = 15; // bit mask: 1 = IRF blocks on 16x16 maps, 4 = also the IRF blocks on 32x32 maps, 2 = head SepConvs run
                      // depthwise + 1x1 as one tcgen05 kernel (pw_tc_kernel<DWK, MW>): bit-identical to the unfused pair,
                      // the depthwise maps are never written.  Round 2: 3.56 -> 3.40 ms / step, -2.3 GB DRAM traffic / step.
                      // 8 = the expand-1 blocks (xif2_2, xif2_3: dw 3x3 -> 1x1 24 -> 24 -> + x) as one CUDA-core kernel
  int pw_ts = 1;      // 1: plain 1x1 GEMMs take their A operand from tensor memory (pw_tc_kernel<0, 16, true>); 0: from shared memory
  int fuse_stem = 1;  // 1: stem + xif1_0 in one kernel (stem_xif1_fused_kernel) when the map tiles by 16x32
  int fuse_irf = 1;   // 1: xif2_0 (expand -> depthwise s2 -> project) as ONE tcgen05 kernel (irf_s2_fused_kernel)
  int dw = 3;  // 3 = auto (default); 0 = one pixel per thread, 1 = register-strip kernel, 2 = rolling-window kernel,
               // 6 = TMA pipeline only where it applies (auto also uses it)
};
static Options g_default_options;
static inline int effective(int impl) { return impl >= 0 ? impl : (tc::available() ? IMPL_TC : IMPL_FFMA); }

struct PwW {
  const float* w = nullptr;  // [cout][cin]
  const float* w_hi = nullptr;  // tf32 split of w for the tcgen05 path: w ~= w_hi + w_lo
  const float* w_lo = nullptr;
  const float* b = nullptr;
  const float* h_w = nullptr;  // host copies (persistent): small layers pass their weights by value
  const float* h_b = nullptr;
  int cin = 0, cout = 0;
};
struct DwW {
  const float* w = nullptr;  // [k*k][c]
  const float* b = nullptr;
  int c = 0, k = 0;
};
struct BlockW {
  PwW pw, pwl;
  DwW dw;
};
struct BranchW {
  DwW enc_dw, corr_dw;
  PwW enc_pw, corr_pw;
};
struct TowerW {
  DwW dw[2];
  PwW pw[2];
};

struct EventPair {
  cudaEvent_t a, b;
  int stage;
};

struct FearContext {
  FsWeights fs;  // host copy of the stem + xif1_0 weights, passed by value to stem_xif1_fused_kernel
  int device = 0;
  Options opt;
  float* d_weights = nullptr;
  float* d_irf_image = nullptr;  // packed shared-memory weights image of the fused xif2_0 kernel
  unsigned long long* d_irf_dbg = nullptr;  // FEAR_IRF_TIMING builds only
  std::vector<float> h_weights;  // host mirror of d_weights (device layout)
  const float *stem_w = nullptr, *stem_b = nullptr;
  BlockW blocks[kNumBlocks];
  PwW neck;
  BranchW branch[2];  // 0 = cls, 1 = reg
  TowerW tower[2];    // 0 = bbox, 1 = cls
  DwW pred_dw[2];     // 0 = bbox, 1 = cls
  const float *pred_w[2] = {nullptr, nullptr}, *pred_b[2] = {nullptr, nullptr};

  int reserved = 0;
  float* ws = nullptr;
  // backbone ping-pong (per frame sizes in floats)
  float *bufX = nullptr, *bufY = nullptr, *bufE = nullptr, *bufD = nullptr;
  // head
  float *hF = nullptr, *hT = nullptr, *hCAT[2] = {nullptr, nullptr}, *hD[2] = {nullptr, nullptr}, *hP = nullptr;
  float* hQ[2] = {nullptr, nullptr};  // tower outputs: [0] = bbox tower (x_reg), [1] = cls tower
  float *zt = nullptr, *mapB = nullptr, *mapC = nullptr;
  float* zu = nullptr;  // dynamic-template (`update`) features of the cls branch, same layout as zt

  int64_t launches = 0;
  int64_t generation = 0;  // bumped whenever workspace pointers or options change (captured CUDA graphs are stale)
  bool profiling = false;
  std::vector<EventPair> events;
  size_t events_used = 0;
  double stage_ms[ST_COUNT] = {0};
  int64_t stage_launches[ST_COUNT] = {0};
};

static constexpr int64_t kActX = 128 * 128 * 16;  // largest block input / output per frame (floats)
static constexpr int64_t kActE = 128 * 128 * 96;  // largest expanded tensor (xif2_0.pw)
static constexpr int64_t kActD = 64 * 64 * 96;    // largest depthwise output (xif2_0.dw)

// RAII bracket around one kernel launch: counts it and, when profiling, records events.
struct LaunchScope {
  FearContext* c;
  cudaStream_t s;
  EventPair* ev = nullptr;
  LaunchScope(FearContext* c_, int stage, cudaStream_t s_) : c(c_), s(s_) {
    if (!c) return;
    c->launches++;
    c->stage_launches[stage]++;
    if (c->profiling && c->events_used < c->events.size()) {
      ev = &c->events[c->events_used++];
      ev->stage = stage;
      cudaEventRecord(ev->a, s);
    }
  }
  ~LaunchScope() {
    if (ev) cudaEventRecord(ev->b, s);
  }
};

static int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_err((int)e, "launch of %s failed: %s", what, cudaGetErrorString(e));
  return 0;
}

// ------------------------------------------------------------------------------ launchers
static int launch_gemm_ffma(FearContext* c, int stage, cudaStream_t s, const float* A, int lda, long long sA,
                            const float* Bw, int ldb, long long sB, const float* bias, const float* R, int ldr,
                            float* C, int ldc, long long sC, int M, int N, int K, int relu, int batch) {
  LaunchScope scope(c, stage, s);
#define GEMM_CASE(TN_)                                                                                    \
  {                                                                                                       \
    dim3 grid((M + 127) / 128, (N + 8 * TN_ - 1) / (8 * TN_), batch);                                     \
    gemm_nt_ffma_kernel<TN_><<<grid, 256, 0, s>>>(A, lda, sA, Bw, ldb, sB, bias, R, ldr, C, ldc, sC, M, N, K, \
                                                  relu);                                                  \
  }
  if (N % 64 == 0) GEMM_CASE(8)
  else if (N % 56 == 0) GEMM_CASE(7)
  else if (N % 48 == 0) GEMM_CASE(6)
  else if (N % 32 == 0) GEMM_CASE(4)
  else if (N % 24 == 0) GEMM_CASE(3)
  else GEMM_CASE(2)
#undef GEMM_CASE
  return check_launch("gemm_nt_ffma_kernel");
}

// 1x1 conv over M pixels: out = act(A * W^T + b (+R)).
static int launch_pw(FearContext* c, int stage, cudaStream_t s, const float* A, int lda, const PwW& w, const float* R,
                     int ldr, float* C, int ldc, int M, int relu) {
  const int pw_impl = effective(c->opt.pw);
  if (pw_impl != IMPL_FFMA && lda == w.cin && ldc == w.cout && (!R || ldr == w.cout) &&
      ((w.cin == 16 && w.cout == 16) || (w.cin == 24 && w.cout == 24))) {
    // streaming layers: one pixel per thread on CUDA cores beats a tensor-core tile pipeline here
    LaunchScope scope(c, stage, s);
    const unsigned blocks = (unsigned)((M + 255) / 256);
    // weights by value in the constant bank (see pw_small_const_kernel)
    if (w.cin == 16) {
      PwSmallWeights<16, 16> pw;
      for (int o = 0; o < 16; ++o)
        for (int k = 0; k < 16; ++k) pw.w[k * 16 + o] = w.h_w[o * 16 + k];
      memcpy(pw.b, w.h_b, sizeof(pw.b));
      pw_small_const_kernel<16, 16><<<blocks, 256, 0, s>>>(A, R, C, M, relu, pw);
    } else {
      PwSmallWeights<24, 24> pw;
      for (int o = 0; o < 24; ++o)
        for (int k = 0; k < 24; ++k) pw.w[k * 24 + o] = w.h_w[o * 24 + k];
      memcpy(pw.b, w.h_b, sizeof(pw.b));
      pw_small_const_kernel<24, 24><<<blocks, 256, 0, s>>>(A, R, C, M, relu, pw);
    }
    return check_launch("pw_small_const_kernel");
  }
  if (pw_impl == IMPL_TC && tc::pw_supported(w.cin, w.cout)) {
    LaunchScope scope(c, stage, s);
    int r = tc::launch_pw(s, A, lda, w.w_hi, w.w_lo, w.b, R, ldr, C, ldc, M, w.cout, w.cin, relu, c->opt.pw_ts != 0);
    if (r) return set_err(r, "tcgen05 pw launch failed (%d)", r);
    return check_launch("tc::pw");
  }
  return launch_gemm_ffma(c, stage, s, A, lda, 0, w.w, w.cin, 0, w.b, R, ldr, C, ldc, 0, M, w.cout, w.cin, relu, 1);
}

static int launch_dw(FearContext* c, int stage, cudaStream_t s, const float* in, const DwW& w, float* out, int B, int H,
                     int W, int stride, bool relu) {
  LaunchScope scope(c, stage, s);
  const int C4 = w.c / 4;
  const int threads = 256;
  const float4* i4 = reinterpret_cast<const float4*>(in);
  const float4* w4 = reinterpret_cast<const float4*>(w.w);
  const float4* b4 = reinterpret_cast<const float4*>(w.b);
  float4* o4 = reinterpret_cast<float4*>(out);
  const bool bias = w.b != nullptr;
  const int Wo = W / stride;
  // TMA-fed shared-memory pipeline (kernels_dw_tma.cuh): stride 1, maps that are multiples of 16x16
  const bool want_tma = (c->opt.dw == 6 || c->opt.dw == 3) && tc::available();
  if (want_tma && stride == 2 && w.k == 5 && relu && bias) {
    // 5x5 stride 2: 8x8 output tiles (19x19 input pixels), 4x1 outputs per thread
    int r = tc::launch_dw_tma_t<5, 2, 8, 8, 4, 1, 4, 2, true, true>(s, in, w.w, w.b, out, B, H, W, w.c, tc::num_sms());
    if (r < 0) return set_err(FEAR_EINVAL, "TMA depthwise launch failed (%d)", r);
    if (r == 0) return check_launch("tc::dw_tma_kernel<5,2>");
  }
  // TMA-fed shared-memory pipeline (kernels_dw_tma.cuh): stride 1, maps that are multiples of 16x16
  if (want_tma && stride == 1 && w.c >= 24) {
    int r = 1;
#define DW_TMA(K_, RELU_, BIAS_) \
  tc::launch_dw_tma_t<K_, 1, 16, 16, 8, 2, 4, 2, RELU_, BIAS_>(s, in, w.w, w.b, out, B, H, W, w.c, tc::num_sms())
    if (w.k == 5 && relu && bias) r = DW_TMA(5, true, true);
    else if (w.k == 3 && relu && bias) r = DW_TMA(3, true, true);
    else if (w.k == 3 && !relu && !bias) r = DW_TMA(3, false, false);
#undef DW_TMA
    if (r < 0) return set_err(FEAR_EINVAL, "TMA depthwise launch failed (%d)", r);
    if (r == 0) return check_launch("tc::dw_tma_kernel");
  }
  const bool want_roll = c->opt.dw == 2 || (c->opt.dw == 3 && w.k == 3 && stride == 1);
  if (want_roll && Wo % 4 == 0 && (H / stride) % 16 == 0) {
    // rolling-window kernels: TX output columns x 16 output rows per thread, weights in registers
    constexpr int ROWS = 16;
    const int Ho = H / stride;
#define ROLL_CASE(K_, S_, TX_, RELU_, BIAS_)                                                        \
  {                                                                                                  \
    const long long total = (long long)B * (Ho / ROWS) * (Wo / TX_) * C4;                            \
    const unsigned blocks = (unsigned)((total + 127) / 128);                                         \
    dw_conv_roll_kernel<K_, S_, TX_, ROWS, RELU_, BIAS_><<<blocks, 128, 0, s>>>(i4, w4, b4, o4, B, H, W, C4); \
  }
    if (w.k == 3 && stride == 1 && relu && bias) ROLL_CASE(3, 1, 4, true, true)
    else if (w.k == 3 && stride == 2 && relu && bias) ROLL_CASE(3, 2, 4, true, true)
    else if (w.k == 5 && stride == 1 && relu && bias) ROLL_CASE(5, 1, 2, true, true)
    else if (w.k == 5 && stride == 2 && relu && bias) ROLL_CASE(5, 2, 2, true, true)
    else if (w.k == 3 && stride == 1 && !relu && !bias) ROLL_CASE(3, 1, 4, false, false)
    else
      return set_err(FEAR_EINVAL, "unsupported depthwise config k=%d s=%d relu=%d bias=%d", w.k, stride, (int)relu,
                     (int)bias);
#undef ROLL_CASE
    return check_launch("dw_conv_roll_kernel");
  }
  if (c->opt.dw == 3 && w.k == 5 && stride == 1 && Wo % 8 == 0 && relu && bias) {
    // 5x5 stride 1: wide strips (fewer loads per FMA: the kernel is bound by L1 wavefronts, not by HBM)
    const long long total = (long long)B * H * (Wo / 8) * C4;
    dw_conv_strip_kernel<5, 1, 8, true, true><<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(
        i4, w4, b4, o4, B, H, W, C4);
    return check_launch("dw_conv_strip_kernel<5,1,8>");
  }
  if (c->opt.dw >= 1 && Wo % 4 == 0) {
    // register-strip kernels: 4 outputs per thread (stride 1) / 2 outputs per thread (stride 2)
    const int TX = stride == 1 ? 4 : 2;
    const long long total = (long long)B * (H / stride) * (Wo / TX) * C4;
    const unsigned blocks = (unsigned)((total + threads - 1) / threads);
    if (w.k == 3 && stride == 1 && relu && bias)
      dw_conv_strip_kernel<3, 1, 4, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
    else if (w.k == 3 && stride == 2 && relu && bias)
      dw_conv_strip_kernel<3, 2, 2, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
    else if (w.k == 5 && stride == 1 && relu && bias)
      dw_conv_strip_kernel<5, 1, 4, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
    else if (w.k == 5 && stride == 2 && relu && bias)
      dw_conv_strip_kernel<5, 2, 2, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
    else if (w.k == 3 && stride == 1 && !relu && !bias)
      dw_conv_strip_kernel<3, 1, 4, false, false><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
    else
      return set_err(FEAR_EINVAL, "unsupported depthwise config k=%d s=%d relu=%d bias=%d", w.k, stride, (int)relu,
                     (int)bias);
    return check_launch("dw_conv_strip_kernel");
  }
  const long long total = (long long)B * (H / stride) * Wo * C4;
  const unsigned blocks = (unsigned)((total + threads - 1) / threads);
  if (w.k == 3 && stride == 1 && relu && bias)
    dw_conv_nhwc_kernel<3, 1, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
  else if (w.k == 3 && stride == 2 && relu && bias)
    dw_conv_nhwc_kernel<3, 2, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
  else if (w.k == 5 && stride == 1 && relu && bias)
    dw_conv_nhwc_kernel<5, 1, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
  else if (w.k == 5 && stride == 2 && relu && bias)
    dw_conv_nhwc_kernel<5, 2, true, true><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
  else if (w.k == 3 && stride == 1 && !relu && !bias)
    dw_conv_nhwc_kernel<3, 1, false, false><<<blocks, threads, 0, s>>>(i4, w4, b4, o4, B, H, W, C4);
  else
    return set_err(FEAR_EINVAL, "unsupported depthwise config k=%d s=%d relu=%d bias=%d", w.k, stride, (int)relu,
                   (int)bias);
  return check_launch("dw_conv_nhwc_kernel");
}

static int launch_transpose(FearContext* c, cudaStream_t s, const float* in, int ldin, long long sIn, float* out,
                            int ldout, long long sOut, int R, int Cn, int batch) {
  LaunchScope scope(c, ST_LAYOUT, s);
  dim3 grid((Cn + 31) / 32, (R + 31) / 32, batch);
  transpose_kernel<<<grid, 256, 0, s>>>(in, ldin, sIn, out, ldout, sOut, R, Cn);
  return check_launch("transpose_kernel");
}

// cat[b, p, 256 + k] = sum_c zt[b, k, c] * cat[b, p, c]    (MobileCorrelation matmul, blocks.py:123)
// `groups` consecutive [B][256][320] buffers starting at cat share the templates (head: cls + reg branch).
static int launch_corr(FearContext* c, const Options& opt, cudaStream_t s, const float* zt, int Bz, float* cat, int B,
                       int groups) {
  const int corr_impl = effective(opt.corr);
  if (corr_impl == IMPL_TC) {
    LaunchScope scope(c, ST_CORR, s);
    int r = tc::launch_corr(s, zt, Bz, cat, B, groups);
    if (r) return set_err(r, "tcgen05 corr launch failed (%d)", r);
    return check_launch("tc::corr");
  }
  for (int g = 0; g < groups; ++g) {
    float* cg = cat + (long long)g * B * kScorePix * kCatC;
    FEAR_TRY(launch_gemm_ffma(c, ST_CORR, s, cg, kCatC, (long long)kScorePix * kCatC, zt, kFeatC,
                              Bz == 1 ? 0 : (long long)kCorrC * kFeatC, nullptr, nullptr, 0, cg + kFeatC, kCatC,
                              (long long)kScorePix * kCatC, kScorePix, kCorrC, kFeatC, 0, B));
  }
  return 0;
}

// ------------------------------------------------------------------------------ executor
// Run backbone blocks [first, last) on NHWC activations X (B frames of h x w), ping-ponging between bufX and bufY
// (bufE = expanded tensor, bufD = depthwise output of the block in flight).  *out receives the output pointer,
// h / w are updated.
static int run_blocks(FearContext* c, cudaStream_t s, float* X, int B, int& h, int& w, int first, int last,
                      float** out) {
  float* Y = (X == c->bufX) ? c->bufY : c->bufX;
  for (int i = first; i < last; ++i) {
    const IrfSpec& sp = kBlocks[i];
    const BlockW& bw = c->blocks[i];
    const int M = B * h * w;
    if (i == 1 && c->opt.fuse_irf && tc::available() && effective(c->opt.pw) == IMPL_TC && c->d_irf_image) {
      // xif2_0: expand 1x1 -> depthwise 3x3 s2 -> project 1x1 in ONE kernel; the expanded tensor stays on the SM
      LaunchScope scope(c, ST_BACKBONE_PW, s);
      int r = tc::launch_irf_s2(s, X, Y, c->d_irf_image, B, h, w, c->d_irf_dbg);
      if (r < 0) return set_err(FEAR_EINVAL, "fused IRF block launch failed (%d)", r);
      if (r == 0) {
        FEAR_TRY(check_launch("tc::irf_s2_fused_kernel"));
        h /= 2;
        w /= 2;
        float* t = X;
        X = Y;
        Y = t;
        continue;
      }
    }
    if ((c->opt.fuse_dwpw & 8) && tc::available() && !sp.has_pw() && sp.stride == 1 && sp.k == 3 && sp.cin == tc::kDpC &&
        sp.cout == tc::kDpC && sp.residual() && bw.dw.b && bw.pwl.h_w && effective(c->opt.pw) != IMPL_FFMA) {
      // expand-1 block: depthwise 3x3 + 1x1 + residual in one kernel (the depthwise map stays in shared memory)
      LaunchScope scope(c, ST_BACKBONE_DW, s);
      PwSmallWeights<tc::kDpC, tc::kDpC> pw;
      for (int o = 0; o < tc::kDpC; ++o)
        for (int k = 0; k < tc::kDpC; ++k) pw.w[k * tc::kDpC + o] = bw.pwl.h_w[o * tc::kDpC + k];
      memcpy(pw.b, bw.pwl.h_b, sizeof(pw.b));
      int r = tc::launch_dw3_pw24(s, X, bw.dw.w, bw.dw.b, pw, Y, B, h, w, tc::num_sms());
      if (r < 0) return set_err(FEAR_EINVAL, "fused depthwise + 24x24 block launch failed (%d)", r);
      if (r == 0) {
        FEAR_TRY(check_launch("tc::dw3_pw24_fused_kernel"));
        float* t = X;
        X = Y;
        Y = t;
        continue;
      }
    }
    const float* E = X;
    if (sp.has_pw()) {
      FEAR_TRY(launch_pw(c, ST_BACKBONE_PW, s, X, sp.cin, bw.pw, nullptr, 0, c->bufE, sp.mid(), M, 1));
      E = c->bufE;
    }
    if ((c->opt.fuse_dwpw & 1) && tc::available() && sp.stride == 1 && sp.has_pw() && w == h &&
        (h == 16 || (h == 32 && (c->opt.fuse_dwpw & 4))) &&
        effective(c->opt.pw) == IMPL_TC) {
      // depthwise + project 1x1 in one tcgen05 kernel (the depthwise map is never written)
      LaunchScope scope(c, ST_BACKBONE_PW, s);
      int r = tc::launch_pw_dw(s, E, B, sp.k, bw.dw.w, bw.dw.b, 1, bw.pwl.w_hi, bw.pwl.w_lo, bw.pwl.b,
                               sp.residual() ? X : nullptr, sp.cout, Y, sp.cout, sp.cout, sp.mid(), 0, h);
      if (r < 0) return set_err(FEAR_EINVAL, "fused depthwise + 1x1 launch failed (%d)", r);
      if (r == 0) {
        FEAR_TRY(check_launch("tc::pw_tc_kernel<DWK>"));
        float* t = X;
        X = Y;
        Y = t;
        continue;
      }
    }
    FEAR_TRY(launch_dw(c, ST_BACKBONE_DW, s, E, bw.dw, c->bufD, B, h, w, sp.stride, true));
    h /= sp.stride;
    w /= sp.stride;
    FEAR_TRY(launch_pw(c, ST_BACKBONE_PW, s, c->bufD, sp.mid(), bw.pwl, sp.residual() ? X : nullptr, sp.cout, Y,
                       sp.cout, B * h * w, 0));
    float* t = X;
    X = Y;
    Y = t;
  }
  *out = X;
  return 0;
}

static StemNorm imagenet_norm() {
  // float32 arithmetic exactly as albumentations.Normalize does it (reference base_tracker.py:73)
  StemNorm n;
  const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
  for (int i = 0; i < 3; ++i) {
    volatile float m = mean[i] * 255.0f, sd = stdv[i] * 255.0f;
    n.mean[i] = m;
    n.inv[i] = 1.0f / sd;
  }
  return n;
}

// img (B,3,H,W) NCHW fp32 -- or raw uint8 (B,H,W,3) with u8 = true -- -> NHWC backbone features
// [B][H/16 * W/16][112] left in *feat (a workspace buffer).
static int run_backbone(FearContext* c, cudaStream_t s, const void* img, int B, int H, int W, const float** feat,
                        bool u8 = false) {
  // (TMA needs 16-byte aligned image rows and base: W % 16 == 0 covers both layouts)
  const bool fuse_stem = c->opt.fuse_stem && tc::available() && (H / 2) % kFsTH == 0 && (W / 2) % kFsTW == 0 &&
                         (reinterpret_cast<uintptr_t>(img) & 15) == 0;
  if (fuse_stem) {
    // stem + xif1_0 (dw3x3 -> 1x1 + residual) in one pass over the image: the block output lands in bufX
    LaunchScope scope(c, ST_STEM, s);
    if (tc::attr_needed(reinterpret_cast<const void*>(stem_xif1_fused_kernel<true>))) {
      CUDA_TRY(cudaFuncSetAttribute(stem_xif1_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFsSmemBytes));
      CUDA_TRY(cudaFuncSetAttribute(stem_xif1_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFsSmemBytes));
    }
    const unsigned blocks = (unsigned)((long long)B * ((H / 2) / kFsTH) * ((W / 2) / kFsTW));
    CUtensorMap tm;
    if (u8) {
      int r = tc::make_tmap_3d(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, img, (uint64_t)3 * W, (uint64_t)H, (uint64_t)B,
                               (uint64_t)3 * W, (uint64_t)3 * W * H, kFsRawPitch, kFsPH, 1);
      if (r) return set_err(FEAR_EINVAL, "tensor map for the uint8 image failed (%d)", r);
      stem_xif1_fused_kernel<true><<<blocks, kFsThreads, kFsSmemBytes, s>>>(tm, c->bufX, H, W, imagenet_norm(), c->fs);
    } else {
      int r = tc::make_tmap_3d(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, img, (uint64_t)W, (uint64_t)H, (uint64_t)3 * B,
                               (uint64_t)W * 4, (uint64_t)W * H * 4, kFsPP, kFsPH, 3);
      if (r) return set_err(FEAR_EINVAL, "tensor map for the float image failed (%d)", r);
      stem_xif1_fused_kernel<false><<<blocks, kFsThreads, kFsSmemBytes, s>>>(tm, c->bufX, H, W, StemNorm(), c->fs);
    }
    FEAR_TRY(check_launch("stem_xif1_fused_kernel"));
  } else {
    LaunchScope scope(c, ST_STEM, s);
    const unsigned blocks = (unsigned)((long long)B * ((H / 2 + 3) / 4) * ((W / 2 + 31) / 32));
    if (u8)
      stem_conv3x3s2_kernel<true><<<blocks, 128, 0, s>>>(static_cast<const uint8_t*>(img), c->stem_w, c->stem_b, c->bufX,
                                                         B, H, W, imagenet_norm());
    else
      stem_conv3x3s2_kernel<false><<<blocks, 128, 0, s>>>(static_cast<const float*>(img), c->stem_w, c->stem_b, c->bufX,
                                                          B, H, W, StemNorm());
    FEAR_TRY(check_launch("stem_conv3x3s2_kernel"));
  }
  int h = H / 2, w = W / 2;
  float* out = nullptr;
  FEAR_TRY(run_blocks(c, s, c->bufX, B, h, w, fuse_stem ? 1 : 0, kNumBlocks, &out));
  *feat = out;
  return 0;
}

// img (B,3,H,W) NCHW -> out NHWC [B][H/16 * W/16][256]   (FEARNet.get_features, fear_net.py:63-66)
static int run_features(FearContext* c, cudaStream_t s, const void* img, int B, int H, int W, float* out,
                        bool u8 = false) {
  const float* X = nullptr;
  FEAR_TRY(run_backbone(c, s, img, B, H, W, &X, u8));
  return launch_pw(c, ST_NECK, s, X, kBackboneC, c->neck, nullptr, 0, out, kFeatC, B * (H / 16) * (W / 16), 0);
}

// F: NHWC search features [B][256][256]; zt: [Bz][64][256]; outputs NCHW maps.
// SepConv of the head (blocks.py:45-72): depthwise 3x3 (no bias, no activation) then 1x1 (+bias, ReLU).
// With the experimental "fuse_dwpw" bit 2 the pair runs as one tcgen05 kernel (the depthwise map is not written).
static int launch_sepconv(FearContext* c, cudaStream_t s, const float* X, const DwW& dw, const PwW& pw, float* out,
                          int ldc, int B) {
  const int M = B * kScorePix;
  if ((c->opt.fuse_dwpw & 2) && tc::available() && effective(c->opt.pw) == IMPL_TC) {
    LaunchScope scope(c, ST_HEAD_PW, s);
    int r = tc::launch_pw_dw(s, X, B, dw.k, dw.w, dw.b, 0, pw.w_hi, pw.w_lo, pw.b, nullptr, 0, out, ldc, pw.cout, pw.cin, 1);
    if (r < 0) return set_err(FEAR_EINVAL, "fused SepConv launch failed (%d)", r);
    if (r == 0) return check_launch("tc::pw_tc_kernel<3>");
  }
  FEAR_TRY(launch_dw(c, ST_HEAD_DW, s, X, dw, c->hT, B, kScore, kScore, 1, false));
  return launch_pw(c, ST_HEAD_PW, s, c->hT, pw.cin, pw, nullptr, 0, out, ldc, M, 1);
}

// zu (optional): dynamic-template features [Bu][64][256] for the classification branch (BoxTower.forward's `update`
// argument, blocks.py:174-179: cls_encode(update, search) -- the regression branch keeps the original template).
static int run_head(FearContext* c, cudaStream_t s, const float* zt, int Bz, const float* F, int B, float* bbox,
                    float* cls, const float* zu = nullptr, int Bu = 0) {
  const int M = B * kScorePix;
  // the two concat buffers are laid out back to back for THIS batch so one correlation launch covers both
  c->hCAT[1] = c->hCAT[0] + (long long)B * kScorePix * kCatC;
  for (int br = 0; br < 2; ++br) {
    const BranchW& w = c->branch[br];
    // MatrixMobile: x -> dw3x3 -> 1x1 (+BN) -> ReLU, written into channels [0,256) of the concat buffer
    FEAR_TRY(launch_sepconv(c, s, F, w.enc_dw, w.enc_pw, c->hCAT[br], kCatC, B));
  }
  // pixel-wise correlation of both branches into channels [256,320) of their concat buffers
  if (zu) {
    FEAR_TRY(launch_corr(c, c->opt, s, zu, Bu, c->hCAT[0], B, 1));  // cls branch <- update template
    FEAR_TRY(launch_corr(c, c->opt, s, zt, Bz, c->hCAT[1], B, 1));  // reg branch <- kernel template
  } else {
    FEAR_TRY(launch_corr(c, c->opt, s, zt, Bz, c->hCAT[0], B, 2));
  }
  for (int br = 0; br < 2; ++br) {
    const BranchW& w = c->branch[br];
    // MobileCorrelation.enc: dw3x3(320) -> 1x1 320->256 (+BN) -> ReLU
    FEAR_TRY(launch_sepconv(c, s, c->hCAT[br], w.corr_dw, w.corr_pw, c->hD[br], kFeatC, B));
  }
  // towers: tower[0] = bbox_tower on reg branch (hD[1]); tower[1] = cls_tower on cls branch (hD[0])
  for (int t = 0; t < 2; ++t) {
    const float* x = c->hD[t == 0 ? 1 : 0];
    float* outs[2] = {c->hP, c->hQ[t]};
    for (int i = 0; i < 2; ++i) {
      FEAR_TRY(launch_sepconv(c, s, x, c->tower[t].dw[i], c->tower[t].pw[i], outs[i], kFeatC, B));
      x = outs[i];
    }
    FEAR_TRY(launch_dw(c, ST_HEAD_DW, s, x, c->pred_dw[t], c->hT, B, kScore, kScore, 1, false));
    LaunchScope scope(c, ST_PRED, s);
    const unsigned blocks = (unsigned)((M * 32 + 255) / 256);
    if (t == 0)
      pred_pw_kernel<4, true><<<blocks, 256, 0, s>>>(c->hT, c->pred_w[0], c->pred_b[0], bbox, B);
    else
      pred_pw_kernel<1, false><<<blocks, 256, 0, s>>>(c->hT, c->pred_w[1], c->pred_b[1], cls, B);
    FEAR_TRY(check_launch("pred_pw_kernel"));
  }
  return 0;
}

static int run_decode(FearContext* c, cudaStream_t s, const float* bbox, const float* cls, int B, int apply_sigmoid,
                      FearBox* boxes) {
  LaunchScope scope(c, ST_DECODE, s);
  decode_kernel<<<B, 256, 0, s>>>(bbox, cls, apply_sigmoid, boxes);
  return check_launch("decode_kernel");
}

// ------------------------------------------------------------------------------ C ABI
// RAII: make the handle's device current for the duration of a C entry point, restore the caller's on exit.
struct DeviceGuard {
  int prev = -1, dev;
  explicit DeviceGuard(int d) : dev(d) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
};

extern "C" int fear_abi_version(void) { return FEAR_ABI_VERSION; }
extern "C" const char* fear_last_error(void) { return g_err; }

// Per-device initialisation; may be called for several devices of one process (each handle remembers its own).
// Leaves `device` current (the reference's `.cuda(cuda_id)` convention); later entry points never change the
// caller's current device.
extern "C" int fear_init(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) return set_err(FEAR_ENODEV, "no CUDA device: %s", cudaGetErrorString(e));
  if (device < 0 || device >= n) return set_err(FEAR_EINVAL, "device %d out of range (%d devices)", device, n);
  cudaDeviceProp p;
  CUDA_TRY(cudaGetDeviceProperties(&p, device));
  if (p.major != 10)
    return set_err(FEAR_ENODEV, "device %d is sm_%d%d; libfear_b200 is built for sm_100a only", device, p.major, p.minor);
  CUDA_TRY(cudaSetDevice(device));
  if (tc::dev_state().inited) return 0;
  return tc::init();
}

extern "C" int fear_weight_count(void) { return (int)weight_table().size(); }
extern "C" const char* fear_weight_name(int i) {
  if (i < 0 || i >= fear_weight_count()) return nullptr;
  return weight_table()[i].name.c_str();
}
extern "C" int64_t fear_weight_numel(int i) {
  if (i < 0 || i >= fear_weight_count()) return -1;
  return weight_table()[i].numel;
}
extern "C" int fear_stage_count(void) { return ST_COUNT; }
extern "C" const char* fear_stage_name(int i) { return (i >= 0 && i < ST_COUNT) ? kStageNames[i] : nullptr; }

extern "C" int fear_pack_weights(const float* blob, const uint64_t* offsets, int n, FearContext** handle) {
  int cur_dev = 0;
  CUDA_TRY(cudaGetDevice(&cur_dev));
  if (!tc::dev_state().inited) return set_err(FEAR_ESTATE, "fear_init() has not been called for device %d", cur_dev);
  if (!blob || !offsets || !handle) return set_err(FEAR_EINVAL, "null argument");
  const auto& table = weight_table();
  if (n != (int)table.size()) return set_err(FEAR_EINVAL, "expected %d tensors, got %d", (int)table.size(), n);
  for (int i = 0; i < n; ++i)
    if ((int64_t)(offsets[i + 1] - offsets[i]) != table[i].numel)
      return set_err(FEAR_EINVAL, "tensor %d (%s): expected %lld elements, got %lld", i, table[i].name.c_str(),
                     (long long)table[i].numel, (long long)(offsets[i + 1] - offsets[i]));

  // Device arena: every tensor 256-byte aligned; depthwise [C][k][k] -> [k*k][C], stem -> [27][16].
  std::vector<float> arena;
  std::vector<size_t> dev_off(n), hi_off(n, 0), lo_off(n, 0);
  auto is_gemm_weight = [&](const std::string& nm) {
    if (nm.rfind("bbox_pred", 0) == 0 || nm.rfind("cls_pred", 0) == 0) return false;
    auto ends = [&](const char* suf) {
      const size_t l = strlen(suf);
      return nm.size() >= l && nm.compare(nm.size() - l, l, suf) == 0;
    };
    return ends(".pw.w") || ends(".pwl.w") || nm == "neck.w";
  };
  for (int i = 0; i < n; ++i) {
    size_t o = (arena.size() + 63) & ~(size_t)63;
    arena.resize(o + table[i].numel, 0.f);
    dev_off[i] = o;
    const float* src = blob + offsets[i];
    const std::string& nm = table[i].name;
    const bool is_dw = nm.size() > 5 && nm.compare(nm.size() - 5, 5, ".dw.w") == 0;
    if (nm == "stem.w") {
      for (int co = 0; co < 16; ++co)
        for (int t = 0; t < 27; ++t) arena[o + t * 16 + co] = src[co * 27 + t];
    } else if (is_dw) {
      // numel = C * kk; kk is 9 or 25.  Find it from the matching bias / table neighbour: C divides numel.
      int kk = 9;
      const bool head = nm.find("xif") == std::string::npos;
      if (!head) {
        for (const IrfSpec& b : kBlocks)
          if (nm == std::string(b.name) + ".dw.w") kk = b.k * b.k;
      }
      const int64_t C = table[i].numel / kk;
      for (int64_t ch = 0; ch < C; ++ch)
        for (int t = 0; t < kk; ++t) arena[o + (int64_t)t * C + ch] = src[ch * kk + t];
    } else {
      memcpy(&arena[o], src, sizeof(float) * table[i].numel);
    }
    if (is_gemm_weight(nm)) {  // tf32 (hi, lo) split for the 3xTF32 tensor-core GEMM
      for (int part = 0; part < 2; ++part) {
        size_t po = (arena.size() + 63) & ~(size_t)63;
        arena.resize(po + table[i].numel, 0.f);
        (part == 0 ? hi_off : lo_off)[i] = po;
        for (int64_t e = 0; e < table[i].numel; ++e) {
          const float hi = tc::host_rna_tf32(src[e]);
          arena[po + e] = part == 0 ? hi : tc::host_rna_tf32(src[e] - hi);
        }
      }
    }
  }
  arena.resize((arena.size() + 63) & ~(size_t)63, 0.f);

  FearContext* c = new FearContext();
  c->device = cur_dev;
  c->opt = g_default_options;
  cudaError_t e = cudaMalloc(&c->d_weights, arena.size() * sizeof(float));
  if (e != cudaSuccess) {
    delete c;
    return set_err(FEAR_ENOMEM, "cudaMalloc(weights) failed: %s", cudaGetErrorString(e));
  }
  e = cudaMemcpy(c->d_weights, arena.data(), arena.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(c->d_weights);
    delete c;
    return set_err((int)e, "cudaMemcpy(weights) failed: %s", cudaGetErrorString(e));
  }
  int idx = 0;
  auto next = [&]() { return (const float*)(c->d_weights + dev_off[idx++]); };
  auto next_pw = [&](PwW& w, int cin, int cout) {  // weight (+ its hi/lo copies) followed by its bias
    w.w_hi = c->d_weights + hi_off[idx];
    w.w_lo = c->d_weights + lo_off[idx];
    w.w = next();
    w.b = next();
    w.h_w = reinterpret_cast<const float*>((w.w - c->d_weights));  // offsets for now; rebased onto h_weights below
    w.h_b = reinterpret_cast<const float*>((w.b - c->d_weights));
    w.cin = cin;
    w.cout = cout;
  };
  c->stem_w = next();
  c->stem_b = next();
  for (int i = 0; i < kNumBlocks; ++i) {
    const IrfSpec& sp = kBlocks[i];
    BlockW& b = c->blocks[i];
    if (sp.has_pw()) next_pw(b.pw, sp.cin, sp.mid());
    b.dw.w = next();
    b.dw.b = next();
    b.dw.c = sp.mid();
    b.dw.k = sp.k;
    next_pw(b.pwl, sp.mid(), sp.cout);
  }
  next_pw(c->neck, kBackboneC, kFeatC);
  for (int br = 0; br < 2; ++br) {
    BranchW& w = c->branch[br];
    w.enc_dw = {next(), nullptr, kFeatC, 3};
    next_pw(w.enc_pw, kFeatC, kFeatC);
    w.corr_dw = {next(), nullptr, kCatC, 3};
    next_pw(w.corr_pw, kCatC, kFeatC);
  }
  for (int t = 0; t < 2; ++t)
    for (int i = 0; i < 2; ++i) {
      c->tower[t].dw[i] = {next(), nullptr, kFeatC, 3};
      next_pw(c->tower[t].pw[i], kFeatC, kFeatC);
    }
  for (int t = 0; t < 2; ++t) {
    c->pred_dw[t] = {next(), nullptr, kFeatC, 3};
    c->pred_w[t] = next();
    c->pred_b[t] = next();
  }
  if (idx != n) {
    cudaFree(c->d_weights);
    delete c;
    return set_err(FEAR_ESTATE, "internal: weight table walk consumed %d of %d tensors", idx, n);
  }
  c->h_weights = std::move(arena);
  {
    auto rebase = [&](PwW& w) {
      w.h_w = c->h_weights.data() + reinterpret_cast<intptr_t>(w.h_w);
      w.h_b = c->h_weights.data() + reinterpret_cast<intptr_t>(w.h_b);
    };
    for (int i = 0; i < kNumBlocks; ++i) {
      if (kBlocks[i].has_pw()) rebase(c->blocks[i].pw);
      rebase(c->blocks[i].pwl);
    }
    rebase(c->neck);
    for (int br = 0; br < 2; ++br) {
      rebase(c->branch[br].enc_pw);
      rebase(c->branch[br].corr_pw);
    }
    for (int t = 0; t < 2; ++t)
      for (int i = 0; i < 2; ++i) rebase(c->tower[t].pw[i]);
  }
  {
    auto host_of = [&](const float* dptr) { return c->h_weights.data() + (dptr - c->d_weights); };
    const BlockW& b0 = c->blocks[0];
    memcpy(c->fs.sw, host_of(c->stem_w), sizeof(c->fs.sw));
    memcpy(c->fs.sb, host_of(c->stem_b), sizeof(c->fs.sb));
    memcpy(c->fs.dw, host_of(b0.dw.w), sizeof(c->fs.dw));
    memcpy(c->fs.db, host_of(b0.dw.b), sizeof(c->fs.db));
    const float* pw = host_of(b0.pwl.w);  // [o][k]
    for (int o = 0; o < 16; ++o)
      for (int k = 0; k < 16; ++k) c->fs.pw[k * 16 + o] = pw[o * 16 + k];
    memcpy(c->fs.pb, host_of(b0.pwl.b), sizeof(c->fs.pb));
    // fused xif2_0 kernel (kernels_irf_fused.cuh): its weights as one shared-memory image
    const BlockW& b1 = c->blocks[1];
    if (kBlocks[1].cin != tc::kIrfCin || kBlocks[1].mid() != tc::kIrfMid || kBlocks[1].cout != tc::kIrfCout ||
        kBlocks[1].k != 3 || kBlocks[1].stride != 2) {
      fear_free(c);
      return set_err(FEAR_ESTATE, "internal: irf_s2_fused_kernel is specialised for xif2_0 (16 -> 96 -> 24, 3x3 s2)");
    }
    std::vector<float> img(tc::kIrfImageFloats);
    tc::irf_build_image(img.data(), host_of(b1.pw.w_hi), host_of(b1.pw.w_lo), host_of(b1.pwl.w_hi), host_of(b1.pwl.w_lo),
                        host_of(b1.dw.w), host_of(b1.pw.b), host_of(b1.dw.b), host_of(b1.pwl.b));
    e = cudaMalloc(&c->d_irf_image, img.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(c->d_irf_image, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      fear_free(c);
      return set_err((int)e, "upload of the fused-block weights failed: %s", cudaGetErrorString(e));
    }
  }
  *handle = c;
  int r = fear_reserve(c, 1);
  if (r) {
    fear_free(c);
    *handle = nullptr;
  }
  return r;
}

extern "C" int fear_reserve(FearContext* c, int max_batch) {
  if (!c) return set_err(FEAR_ESTATE, "null handle");
  if (max_batch < 1) return set_err(FEAR_EINVAL, "max_batch must be >= 1");
  if (max_batch <= c->reserved) return 0;
  DeviceGuard guard(c->device);
  CUDA_TRY(cudaDeviceSynchronize());
  if (c->ws) cudaFree(c->ws);
  c->ws = nullptr;
  c->reserved = 0;
  const int64_t per_frame[] = {
      kActX, kActX, kActE, kActD,                                   // bufX bufY bufE bufD
      (int64_t)kScorePix * kFeatC,                                  // hF
      (int64_t)kScorePix * kCatC,                                   // hT
      (int64_t)kScorePix * kCatC, (int64_t)kScorePix * kCatC,       // hCAT[2]
      (int64_t)kScorePix * kFeatC, (int64_t)kScorePix * kFeatC,     // hD[2]
      (int64_t)kScorePix * kFeatC,                                  // hP
      (int64_t)kScorePix * kFeatC, (int64_t)kScorePix * kFeatC,     // hQ[2]
      (int64_t)kTmplPix * kFeatC,                                   // zt
      4 * kScorePix, kScorePix,                                     // mapB mapC
      (int64_t)kTmplPix * kFeatC,                                   // zu
  };
  int64_t total = 0;
  std::vector<int64_t> offs;
  for (int64_t pf : per_frame) {
    offs.push_back(total);
    total += ((pf * max_batch + 63) / 64) * 64;
  }
  cudaError_t e = cudaMalloc(&c->ws, (size_t)total * sizeof(float));
  if (e != cudaSuccess)
    return set_err(FEAR_ENOMEM, "workspace cudaMalloc(%lld MB) failed: %s", (long long)(total * 4 >> 20),
                   cudaGetErrorString(e));
  float* p = c->ws;
  c->bufX = p + offs[0];
  c->bufY = p + offs[1];
  c->bufE = p + offs[2];
  c->bufD = p + offs[3];
  c->hF = p + offs[4];
  c->hT = p + offs[5];
  c->hCAT[0] = p + offs[6];
  c->hCAT[1] = p + offs[7];
  c->hD[0] = p + offs[8];
  c->hD[1] = p + offs[9];
  c->hP = p + offs[10];
  c->hQ[0] = p + offs[11];
  c->hQ[1] = p + offs[12];
  c->zt = p + offs[13];
  c->mapB = p + offs[14];
  c->mapC = p + offs[15];
  c->zu = p + offs[16];
  c->generation++;
  c->reserved = max_batch;
  return 0;
}

extern "C" void fear_free(FearContext* c) {
  if (!c) return;
  DeviceGuard guard(c->device);
  cudaDeviceSynchronize();
  for (auto& ev : c->events) {
    cudaEventDestroy(ev.a);
    cudaEventDestroy(ev.b);
  }
  if (c->ws) cudaFree(c->ws);
  if (c->d_weights) cudaFree(c->d_weights);
  if (c->d_irf_image) cudaFree(c->d_irf_image);
  delete c;
}

static int check_ctx(FearContext* c) {
  if (!c || !c->d_weights || !c->ws) return set_err(FEAR_ESTATE, "handle not initialised");
  return 0;
}

extern "C" int fear_get_features(FearContext* c, const float* d_img, int B, int H, int W, float* d_feat, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_img || !d_feat || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (H % 16 || W % 16 || H < 16 || W < 16 || H > 256 || W > 256)
    return set_err(FEAR_EINVAL, "H, W must be multiples of 16 in [16, 256] (got %dx%d)", H, W);
  cudaStream_t s = (cudaStream_t)stream;
  const int P = (H / 16) * (W / 16);
  for (int b0 = 0; b0 < B; b0 += c->reserved) {
    const int nb = (B - b0 < c->reserved) ? B - b0 : c->reserved;
    FEAR_TRY(run_features(c, s, d_img + (long long)b0 * 3 * H * W, nb, H, W, c->hF));
    FEAR_TRY(launch_transpose(c, s, c->hF, kFeatC, (long long)P * kFeatC, d_feat + (long long)b0 * kFeatC * P, P,
                              (long long)kFeatC * P, P, kFeatC, nb));
  }
  return 0;
}

extern "C" int fear_backbone(FearContext* c, const float* d_img, int B, int H, int W, float* d_feat, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_img || !d_feat || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (H % 16 || W % 16 || H < 16 || W < 16 || H > 256 || W > 256)
    return set_err(FEAR_EINVAL, "H, W must be multiples of 16 in [16, 256] (got %dx%d)", H, W);
  cudaStream_t s = (cudaStream_t)stream;
  const int P = (H / 16) * (W / 16);
  for (int b0 = 0; b0 < B; b0 += c->reserved) {
    const int nb = (B - b0 < c->reserved) ? B - b0 : c->reserved;
    const float* X = nullptr;
    FEAR_TRY(run_backbone(c, s, d_img + (long long)b0 * 3 * H * W, nb, H, W, &X));
    FEAR_TRY(launch_transpose(c, s, X, kBackboneC, (long long)P * kBackboneC, d_feat + (long long)b0 * kBackboneC * P,
                              P, (long long)kBackboneC * P, P, kBackboneC, nb));
  }
  return 0;
}

// zfeat NCHW (Bz,256,8,8) -> c->zt chunk [nz][64][256]
static int stage_template(FearContext* c, cudaStream_t s, const float* d_zfeat, int nz) {
  return launch_transpose(c, s, d_zfeat, kTmplPix, (long long)kFeatC * kTmplPix, c->zt, kFeatC,
                          (long long)kTmplPix * kFeatC, kFeatC, kTmplPix, nz);
}

// zfeat NCHW (n,256,8,8) -> dst chunk [n][64][256]
static int stage_template_to(FearContext* c, cudaStream_t s, const float* d_zfeat, int nz, float* dst) {
  return launch_transpose(c, s, d_zfeat, kTmplPix, (long long)kFeatC * kTmplPix, dst, kFeatC,
                          (long long)kTmplPix * kFeatC, kFeatC, kTmplPix, nz);
}

extern "C" int fear_head_update(FearContext* c, const float* d_zfeat, int Bz, const float* d_zupdate, int Bu,
                                const float* d_xfeat, int B, float* d_bbox, float* d_cls, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_zfeat || !d_xfeat || !d_bbox || !d_cls || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (Bz != 1 && Bz != B) return set_err(FEAR_EINVAL, "template batch must be 1 or B (got %d vs %d)", Bz, B);
  if (d_zupdate && Bu != 1 && Bu != B)
    return set_err(FEAR_EINVAL, "update-template batch must be 1 or B (got %d vs %d)", Bu, B);
  cudaStream_t s = (cudaStream_t)stream;
  if (Bz == 1) FEAR_TRY(stage_template(c, s, d_zfeat, 1));
  if (d_zupdate && Bu == 1) FEAR_TRY(stage_template_to(c, s, d_zupdate, 1, c->zu));
  for (int b0 = 0; b0 < B; b0 += c->reserved) {
    const int nb = (B - b0 < c->reserved) ? B - b0 : c->reserved;
    if (Bz != 1) FEAR_TRY(stage_template(c, s, d_zfeat + (long long)b0 * kFeatC * kTmplPix, nb));
    if (d_zupdate && Bu != 1)
      FEAR_TRY(stage_template_to(c, s, d_zupdate + (long long)b0 * kFeatC * kTmplPix, nb, c->zu));
    FEAR_TRY(launch_transpose(c, s, d_xfeat + (long long)b0 * kFeatC * kScorePix, kScorePix,
                              (long long)kFeatC * kScorePix, c->hF, kFeatC, (long long)kScorePix * kFeatC, kFeatC,
                              kScorePix, nb));
    FEAR_TRY(run_head(c, s, c->zt, Bz == 1 ? 1 : nb, c->hF, nb, d_bbox + (long long)b0 * 4 * kScorePix,
                      d_cls + (long long)b0 * kScorePix, d_zupdate ? c->zu : nullptr, Bu == 1 ? 1 : nb));
  }
  return 0;
}

extern "C" int fear_head(FearContext* c, const float* d_zfeat, int Bz, const float* d_xfeat, int B, float* d_bbox,
                         float* d_cls, void* stream) {
  return fear_head_update(c, d_zfeat, Bz, nullptr, 0, d_xfeat, B, d_bbox, d_cls, stream);
}

static int track_impl(FearContext* c, cudaStream_t s, const float* d_template, const void* d_search,
                      const float* d_zfeat, int Bz, int B, float* d_bbox, float* d_cls, FearBox* d_boxes,
                      bool search_u8 = false) {
  if (d_zfeat && Bz == 1) FEAR_TRY(stage_template(c, s, d_zfeat, 1));
  for (int b0 = 0; b0 < B; b0 += c->reserved) {
    const int nb = (B - b0 < c->reserved) ? B - b0 : c->reserved;
    int nz = nb;
    if (d_template) {
      // template branch writes NHWC [nb][64][256] straight into zt (= the correlation kernel's layout)
      FEAR_TRY(run_features(c, s, d_template + (long long)b0 * 3 * 128 * 128, nb, 128, 128, c->zt));
    } else if (Bz != 1) {
      FEAR_TRY(stage_template(c, s, d_zfeat + (long long)b0 * kFeatC * kTmplPix, nb));
    } else {
      nz = 1;
    }
    const void* sp = search_u8 ? (const void*)(static_cast<const uint8_t*>(d_search) + (long long)b0 * 3 * 256 * 256)
                               : (const void*)(static_cast<const float*>(d_search) + (long long)b0 * 3 * 256 * 256);
    FEAR_TRY(run_features(c, s, sp, nb, 256, 256, c->hF, search_u8));
    float* bb = d_bbox ? d_bbox + (long long)b0 * 4 * kScorePix : c->mapB;
    float* cc = d_cls ? d_cls + (long long)b0 * kScorePix : c->mapC;
    FEAR_TRY(run_head(c, s, c->zt, nz, c->hF, nb, bb, cc));
    if (d_boxes) FEAR_TRY(run_decode(c, s, bb, cc, nb, 1, d_boxes + b0));
  }
  return 0;
}

extern "C" int fear_track(FearContext* c, const float* d_search, const float* d_zfeat, int Bz, int B, float* d_bbox,
                          float* d_cls, FearBox* d_boxes, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_search || !d_zfeat || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (Bz != 1 && Bz != B) return set_err(FEAR_EINVAL, "template batch must be 1 or B (got %d vs %d)", Bz, B);
  if (!d_boxes && (!d_bbox || !d_cls)) return set_err(FEAR_EINVAL, "no output requested");
  return track_impl(c, (cudaStream_t)stream, nullptr, d_search, d_zfeat, Bz, B, d_bbox, d_cls, d_boxes);
}

extern "C" int fear_track_u8(FearContext* c, const uint8_t* d_search_u8, const float* d_zfeat, int Bz, int B,
                             float* d_bbox, float* d_cls, FearBox* d_boxes, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_search_u8 || !d_zfeat || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (Bz != 1 && Bz != B) return set_err(FEAR_EINVAL, "template batch must be 1 or B (got %d vs %d)", Bz, B);
  if (!d_boxes && (!d_bbox || !d_cls)) return set_err(FEAR_EINVAL, "no output requested");
  return track_impl(c, (cudaStream_t)stream, nullptr, d_search_u8, d_zfeat, Bz, B, d_bbox, d_cls, d_boxes, true);
}

extern "C" int fear_get_features_u8(FearContext* c, const uint8_t* d_img_u8, int B, int H, int W, float* d_feat,
                                    void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_img_u8 || !d_feat || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (H % 16 || W % 16 || H < 16 || W < 16 || H > 256 || W > 256)
    return set_err(FEAR_EINVAL, "H, W must be multiples of 16 in [16, 256] (got %dx%d)", H, W);
  cudaStream_t s = (cudaStream_t)stream;
  const int P = (H / 16) * (W / 16);
  for (int b0 = 0; b0 < B; b0 += c->reserved) {
    const int nb = (B - b0 < c->reserved) ? B - b0 : c->reserved;
    FEAR_TRY(run_features(c, s, d_img_u8 + (long long)b0 * 3 * H * W, nb, H, W, c->hF, true));
    FEAR_TRY(launch_transpose(c, s, c->hF, kFeatC, (long long)P * kFeatC, d_feat + (long long)b0 * kFeatC * P, P,
                              (long long)kFeatC * P, P, kFeatC, nb));
  }
  return 0;
}

extern "C" int fear_forward(FearContext* c, const float* d_template, const float* d_search, int B, float* d_bbox,
                            float* d_cls, FearBox* d_boxes, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_template || !d_search || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (!d_boxes && (!d_bbox || !d_cls)) return set_err(FEAR_EINVAL, "no output requested");
  return track_impl(c, (cudaStream_t)stream, d_template, d_search, nullptr, B, B, d_bbox, d_cls, d_boxes);
}

// Context crop + padding + bilinear resize on the device (get_extended_crop of the tracking loop; see
// crop_resize_u8_kernel).  d_params: 8 + 6 * out_size int32 (layout in kernels_ffma.cuh / include/fear_b200.h).
extern "C" int fear_crop_resize_u8(const uint8_t* d_frame, int H, int W, const int32_t* d_params, uint8_t* d_crop,
                                   int out_size, void* stream) {
  if (!d_frame || !d_params || !d_crop || H < 1 || W < 1 || out_size < 1 || out_size > 1024)
    return set_err(FEAR_EINVAL, "bad argument");
  const int n = out_size * out_size;
  crop_resize_u8_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_frame, H, W, d_params, d_crop, out_size);
  return check_launch("crop_resize_u8_kernel");
}

// N context crops for N tracks in one launch, context boxes and resize coefficients derived on the device from the
// tracks' boxes (kernels_multitrack.cuh).
extern "C" int fear_track_crops_u8(const FearFrame* d_frames, int F, const int32_t* d_frame_of_track, FearTrack* d_tracks,
                                   int N, int out_size, double context, uint8_t* d_crops, void* stream) {
  if (!d_frames || !d_frame_of_track || !d_tracks || !d_crops || F < 1 || N < 1 || N > 65535 || out_size < 1 ||
      out_size > 1024 || !(context >= 0.0 && context <= 1e6))
    return set_err(FEAR_EINVAL, "bad argument");
  const dim3 grid((out_size * out_size + 255) / 256, N);
  track_crops_u8_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_frames, F, d_frame_of_track, d_tracks, out_size,
                                                                context, d_crops);
  return check_launch("track_crops_u8_kernel");
}

// Decoded box records -> next box of every live track (rescale_bbox + clamp_bbox on the device).
extern "C" int fear_track_advance(const FearBox* d_boxes, const FearFrame* d_frames, const int32_t* d_frame_of_track,
                                  FearTrack* d_tracks, int N, int instance_size, void* stream) {
  if (!d_boxes || !d_frames || !d_frame_of_track || !d_tracks || N < 1 || instance_size < 1)
    return set_err(FEAR_EINVAL, "bad argument");
  track_advance_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(d_boxes, d_frames, d_frame_of_track,
                                                                           d_tracks, N, instance_size);
  return check_launch("track_advance_kernel");
}

extern "C" int fear_decode(const float* d_bbox, const float* d_cls, int B, int apply_sigmoid, FearBox* d_boxes,
                           void* stream) {
  if (!d_bbox || !d_cls || !d_boxes || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  return run_decode(nullptr, (cudaStream_t)stream, d_bbox, d_cls, B, apply_sigmoid, d_boxes);
}

extern "C" int fear_corr_nhwc_f32(const float* d_zt, int Bz, float* d_cat, int B, void* stream) {
  if (!d_zt || !d_cat || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (Bz != 1 && Bz != B) return set_err(FEAR_EINVAL, "template batch must be 1 or B (got %d vs %d)", Bz, B);
  if (!tc::dev_state().inited) return set_err(FEAR_ESTATE, "fear_init() has not been called for the current device");
  return launch_corr(nullptr, g_default_options, (cudaStream_t)stream, d_zt, Bz, d_cat, B, 1);
}

extern "C" size_t fear_corr_concat_workspace_bytes(int B, int Bz) {
  if (B < 1 || Bz < 1) return 0;
  return ((size_t)B * kScorePix * kCatC + (size_t)Bz * kCorrC * kFeatC) * sizeof(float);
}

// NCHW in / NCHW out through the hot path's channels-last tcgen05 kernel; the two layout changes use the
// caller's workspace (nothing is allocated, the stream is never synchronised).
extern "C" int fear_corr_concat_ws_f32(const float* d_z, int Bz, const float* d_x, int B, float* d_out, void* d_workspace,
                                       size_t workspace_bytes, void* stream) {
  if (!d_z || !d_x || !d_out || !d_workspace || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (Bz != 1 && Bz != B) return set_err(FEAR_EINVAL, "template batch must be 1 or B (got %d vs %d)", Bz, B);
  if (workspace_bytes < fear_corr_concat_workspace_bytes(B, Bz) || (reinterpret_cast<uintptr_t>(d_workspace) & 1023))
    return set_err(FEAR_EINVAL, "workspace must be 1024-byte aligned and hold fear_corr_concat_workspace_bytes(B, Bz) = %zu bytes",
                   fear_corr_concat_workspace_bytes(B, Bz));
  if (!tc::dev_state().inited) return set_err(FEAR_ESTATE, "fear_init() has not been called for the current device");
  cudaStream_t s = (cudaStream_t)stream;
  float* cat = static_cast<float*>(d_workspace);
  float* zt = cat + (size_t)B * kScorePix * kCatC;
  // z [c][k] -> zt [k][c];  x [c][p] -> cat[p][0:256]
  FEAR_TRY(launch_transpose(nullptr, s, d_z, kCorrC, (long long)kFeatC * kCorrC, zt, kFeatC, (long long)kCorrC * kFeatC,
                            kFeatC, kCorrC, Bz));
  FEAR_TRY(launch_transpose(nullptr, s, d_x, kScorePix, (long long)kFeatC * kScorePix, cat, kCatC,
                            (long long)kScorePix * kCatC, kFeatC, kScorePix, B));
  FEAR_TRY(launch_corr(nullptr, g_default_options, s, zt, Bz, cat, B, 1));
  // cat [p][320] -> out [320][p]
  return launch_transpose(nullptr, s, cat, kCatC, (long long)kScorePix * kCatC, d_out, kScorePix,
                          (long long)kCatC * kScorePix, kScorePix, kCatC, B);
}

// Workspace-free form with the signature SURVEY.md 8(b) lists: a direct CUDA-core kernel on the reference's own
// layouts (compatibility entry point -- the hot path and the _ws form above use the tcgen05 kernel).
extern "C" int fear_corr_concat_f32(const float* d_z, int Bz, const float* d_x, int B, float* d_out, void* stream) {
  if (!d_z || !d_x || !d_out || B < 1) return set_err(FEAR_EINVAL, "bad argument");
  if (Bz != 1 && Bz != B) return set_err(FEAR_EINVAL, "template batch must be 1 or B (got %d vs %d)", Bz, B);
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaMemcpy2DAsync(d_out, (size_t)kCatC * kScorePix * sizeof(float), d_x, (size_t)kFeatC * kScorePix * sizeof(float),
                             (size_t)kFeatC * kScorePix * sizeof(float), (size_t)B, cudaMemcpyDeviceToDevice, s));
  corr_nchw_ffma_kernel<<<dim3(kScorePix / 64, B), 256, 0, s>>>(d_z, Bz == 1 ? 0ll : (long long)kFeatC * kCorrC, d_x, d_out);
  return check_launch("corr_nchw_ffma_kernel");
}

// ---- debug / introspection of intermediates (tests localise a mismatch with these) ----------
extern "C" int fear_debug_backbone_prefix(FearContext* c, const float* d_img, int B, int H, int W, int nblocks,
                                          float* d_out, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!d_img || !d_out || B < 1 || B > c->reserved || nblocks < 0 || nblocks > kNumBlocks)
    return set_err(FEAR_EINVAL, "bad argument (B must be <= reserved batch)");
  cudaStream_t s = (cudaStream_t)stream;
  {
    LaunchScope scope(c, ST_STEM, s);
    const unsigned blocks = (unsigned)((long long)B * ((H / 2 + 3) / 4) * ((W / 2 + 31) / 32));
    stem_conv3x3s2_kernel<false><<<blocks, 128, 0, s>>>(d_img, c->stem_w, c->stem_b, c->bufX, B, H, W, StemNorm());
    FEAR_TRY(check_launch("stem_conv3x3s2_kernel"));
  }
  int h = H / 2, w = W / 2;
  float* X = nullptr;
  FEAR_TRY(run_blocks(c, s, c->bufX, B, h, w, 0, nblocks, &X));
  const int ch = nblocks ? kBlocks[nblocks - 1].cout : kStemC;
  const int P = h * w;
  return launch_transpose(c, s, X, ch, (long long)P * ch, d_out, P, (long long)ch * P, P, ch, B);
}

// Copy a head intermediate of the LAST run (first B frames) out as NCHW (B, C, 16, 16).
extern "C" int fear_debug_head_tensor(FearContext* c, const char* name, int B, float* d_out, void* stream) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (!name || !d_out || B < 1 || B > c->reserved) return set_err(FEAR_EINVAL, "bad argument");
  const float* src = nullptr;
  int ch = kFeatC;
  if (!strcmp(name, "cat_cls")) src = c->hCAT[0], ch = kCatC;
  else if (!strcmp(name, "cat_reg")) src = c->hCAT[1], ch = kCatC;
  else if (!strcmp(name, "cls_dw")) src = c->hD[0];
  else if (!strcmp(name, "reg_dw")) src = c->hD[1];
  else if (!strcmp(name, "x_reg")) src = c->hQ[0];
  else if (!strcmp(name, "cls_tower")) src = c->hQ[1];
  else if (!strcmp(name, "search_features")) src = c->hF;
  else return set_err(FEAR_EINVAL, "unknown head tensor '%s'", name);
  return launch_transpose(c, (cudaStream_t)stream, src, ch, (long long)kScorePix * ch, d_out, kScorePix,
                          (long long)ch * kScorePix, kScorePix, ch, B);
}

extern "C" int fear_set_option(FearContext* c, const char* key, const char* value) {
  if (!key || !value) return set_err(FEAR_EINVAL, "null option");
  Options& o = c ? c->opt : g_default_options;
  if (c) c->generation++;
  if (!strcmp(key, "pdl")) {  // process-wide: programmatic dependent launch for the TMA / tcgen05 kernels
    tc::pdl_enabled() = atoi(value) != 0;
    return 0;
  }
  if (!strcmp(key, "fuse_dwpw")) {
    o.fuse_dwpw = atoi(value) & 15;  // bit 0: 16x16-stage backbone blocks, bit 1: the head's SepConvs, bit 2: also the 32x32-stage blocks, bit 3: expand-1 blocks
    return 0;
  }
  if (!strcmp(key, "pw_ts")) {
    o.pw_ts = atoi(value) != 0;
    return 0;
  }
  if (!strcmp(key, "fuse_stem")) {
    o.fuse_stem = atoi(value) != 0;
    return 0;
  }
  if (!strcmp(key, "fuse_irf")) {
    o.fuse_irf = atoi(value) != 0;
    return 0;
  }
  if (!strcmp(key, "dw")) {
    if (!strcmp(value, "pixel")) o.dw = 0;
    else if (!strcmp(value, "strip")) o.dw = 1;
    else if (!strcmp(value, "roll")) o.dw = 2;
    else if (!strcmp(value, "auto")) o.dw = 3;  // measured best per shape: TMA pipeline where it applies, else rolling window (3x3 s1) / register strip
    else if (!strcmp(value, "tma")) o.dw = 6;
    else return set_err(FEAR_EINVAL, "unknown depthwise implementation '%s' (pixel | strip | roll | tma | auto)", value);
    return 0;
  }
  int impl;
  if (!strcmp(value, "ffma")) impl = IMPL_FFMA;
  else if (!strcmp(value, "tcgen05")) impl = IMPL_TC;
  else if (!strcmp(value, "auto")) impl = -1;
  else return set_err(FEAR_EINVAL, "unknown implementation '%s' (auto | ffma | tcgen05)", value);
  if (impl > IMPL_FFMA && !tc::available()) return set_err(FEAR_EINVAL, "tcgen05 kernels not available in this build");
  if (!strcmp(key, "corr")) o.corr = impl;
  else if (!strcmp(key, "pw")) o.pw = impl;
  else return set_err(FEAR_EINVAL, "unknown option '%s' (corr | pw)", key);
  return 0;
}

#ifdef FEAR_IRF_TIMING
// Profiling build only (python -m feartracker_b200.build with FEAR_NVCC_FLAGS=-DFEAR_IRF_TIMING; not declared in the
// public header): per-warp cycle counters of the last irf_s2_fused_kernel launch, [148][8 warps][8] uint64.
extern "C" int fear_debug_irf_timing(FearContext* c, unsigned long long* host_out, int n) {
  if (!c || !host_out) return FEAR_EINVAL;
  DeviceGuard guard(c->device);
  if (!c->d_irf_dbg) {
    CUDA_TRY(cudaMalloc(&c->d_irf_dbg, 148 * 128 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(c->d_irf_dbg, 0, 148 * 128 * sizeof(unsigned long long)));
    return 1;  // armed: run a step, then call again
  }
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(host_out, c->d_irf_dbg, sizeof(unsigned long long) * (n < 148 * 128 ? n : 148 * 128), cudaMemcpyDeviceToHost));
  return 0;
}
#endif

#ifdef FEAR_CORR_ABLATE
// Profiling build only (FEAR_NVCC_FLAGS=-DFEAR_CORR_ABLATE; not in the public header): roles of corr_ts_kernel that skip
// their work.  1 = MMAs, 2 = convert, 4 = epilogue, 8 = x tiles re-read from L2 (no HBM stream).  Results are garbage.
extern "C" int fear_debug_corr_ablate(int mask) {
  CUDA_TRY(cudaMemcpyToSymbol(tc::g_corr_ablate, &mask, sizeof(int)));
  return 0;
}
#endif

#ifdef FEAR_PW_ABLATE
// Profiling build only (FEAR_NVCC_FLAGS=-DFEAR_PW_ABLATE): see kernels_tc.cuh / tools/pw_ablate.py.
extern "C" int fear_debug_pw_ablate(int mask) {
  CUDA_TRY(cudaMemcpyToSymbol(tc::g_pw_ablate, &mask, sizeof(int)));
  return 0;
}
#endif

#ifdef FEAR_PW_TIMING
// Profiling build only (FEAR_NVCC_FLAGS=-DFEAR_PW_TIMING): per-launch role cycle counters of pw_tc_kernel since the last
// call (launch ordinal modulo 64); counters [64][32] u64, info [64][8] int.  Resets both.  tools/pw_timing.py
extern "C" int fear_debug_pw_timing(unsigned long long* counters, int* info) {
  CUDA_TRY(cudaDeviceSynchronize());
  if (counters) CUDA_TRY(cudaMemcpyFromSymbol(counters, tc::g_pw_timing, sizeof(unsigned long long) * 64 * 32));
  if (info) memcpy(info, tc::pw_timing_info(), sizeof(tc::PwTimingInfo) * 64);
  static unsigned long long zeros[64 * 32];
  CUDA_TRY(cudaMemcpyToSymbol(tc::g_pw_timing, zeros, sizeof(zeros)));
  int n = tc::pw_timing_next();
  tc::pw_timing_next() = 0;
  return n;
}
#endif

extern "C" int64_t fear_launch_count(const FearContext* c) { return c ? c->launches : 0; }
extern "C" int64_t fear_generation(const FearContext* c) { return c ? c->generation : -1; }

extern "C" int fear_profile(FearContext* c, int enable) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (enable && c->events.empty()) {
    c->events.resize(8192);
    for (auto& ev : c->events) {
      CUDA_TRY(cudaEventCreate(&ev.a));
      CUDA_TRY(cudaEventCreate(&ev.b));
    }
  }
  c->profiling = enable != 0;
  c->events_used = 0;
  for (int i = 0; i < ST_COUNT; ++i) {
    c->stage_ms[i] = 0;
    c->stage_launches[i] = 0;
  }
  return 0;
}

extern "C" int fear_stage_ms(FearContext* c, int i, float* ms, int64_t* launches) {
  FEAR_TRY(check_ctx(c));
  DeviceGuard guard(c->device);
  if (i < 0 || i >= ST_COUNT) return set_err(FEAR_EINVAL, "stage index out of range");
  if (c->events_used) {
    CUDA_TRY(cudaDeviceSynchronize());
    for (size_t k = 0; k < c->events_used; ++k) {
      float t = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&t, c->events[k].a, c->events[k].b));
      c->stage_ms[c->events[k].stage] += t;
    }
    c->events_used = 0;
  }
  if (ms) *ms = (float)c->stage_ms[i];
  if (launches) *launches = c->stage_launches[i];
  return 0;
}
