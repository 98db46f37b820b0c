// C-ABI launchers for the tcgen05 GEMM / implicit-GEMM convolution kernel (see gemm.cuh).
#include "gemm.cuh"
#include "host_utils.h"
#include "../../include/passl_b200.h"

#include <string.h>

#include <functional>
#include <mutex>

namespace pb {

// 128 x 128 bf16 identity used as the A operand of the residual-through-the-tensor-pipe iterations (gemm.cuh, res_iters)
__device__ __nv_bfloat16 g_eye128[128 * 128];
__global__ void eye128_init_kernel() {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 128 * 128) g_eye128[i] = __float2bfloat16_rn((i / 128) == (i % 128) ? 1.f : 0.f);
}
static int eye128_ptr(const void** out, cudaStream_t st) {
  static void* ptr = nullptr;
  if (!ptr) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    PB_CUDA_CHECK(cudaStreamIsCapturing(st, &cs));
    if (cs != cudaStreamCaptureStatusNone) { *out = nullptr; return PB_OK; }   // cannot initialise inside a capture: epilogue path
    PB_CUDA_CHECK(cudaGetSymbolAddress(&ptr, g_eye128));
    eye128_init_kernel<<<64, 256, 0, st>>>();
    PB_LAUNCH_CHECK();
    PB_CUDA_CHECK(cudaStreamSynchronize(st));     // once per process: later launches may come from other streams
  }
  *out = ptr;
  return PB_OK;
}

// route the residual through the MMA when the epilogue semantics allow it (out = A.B + bias + residual, bf16, plain row-major)
static int setup_residual_mma(GemmParams& p, const void* residual, long long ldc, cudaStream_t st) {
  p.res_iters = 0;
  if (!residual || p.out_fp32 || p.out_pixel || p.act != ACT_NONE || p.alpha != 1.f || p.aux || p.preact || p.splits != 1 ||
      p.n_blocks_per_tap > 0 || (reinterpret_cast<uintptr_t>(residual) & 15))
    return PB_OK;
  const void* eye = nullptr;
  int rc = eye128_ptr(&eye, st);
  if (rc) return rc;
  if (!eye) return PB_OK;
  uint64_t ed[2] = {128, 128}, es[1] = {256};
  uint32_t eb[2] = {64, 128};
  rc = make_tmap_bf16(&p.eye_map, eye, 2, ed, es, eb);
  if (rc) return rc;
  uint64_t rd[2] = {(uint64_t)p.N, (uint64_t)p.M}, rs[1] = {(uint64_t)ldc * 2};
  uint32_t rb[2] = {64, 64};
  rc = make_tmap_bf16(&p.res_map, residual, 2, rd, rs, rb);
  if (rc) return rc;
  p.res_iters = 2;
  return PB_OK;
}

template <int BN, int BK, bool A_MN, bool B_MN, int EPI = 0, int CG = 1, bool HALO = false, int EW = kEpiWarps>
static int launch_gemm_t(const GemmParams& p, cudaStream_t st) {
  using S = GemmSmem<BN, BK, A_MN, B_MN, EPI, CG, HALO, EW>;
  auto kern = gemm_tcgen05_kernel<BN, BK, A_MN, B_MN, EPI, CG, HALO, EW>;
  constexpr int kThreads = 64 + 32 * EW;
  static bool attr_set = false;
  if (!attr_set) {
    PB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    attr_set = true;
  }
  int tiles = (CG == 2 ? (p.m_blocks + 1) / 2 : p.m_blocks) * p.n_blocks * p.splits;
  int slots = num_sms() / CG;
  int grid = (tiles < slots ? tiles : slots) * CG;
  if (grid <= 0) return PB_OK;
  if (p.col_sum) {
    if (p.out_fp32 || p.n_blocks_per_tap > 0 || p.splits != 1) return PB_ERR_UNSUPPORTED;
    PB_CUDA_CHECK(cudaMemsetAsync(p.col_sum, 0, (size_t)num_sms() * 4 * 2 * p.N * sizeof(float), st));
  }
  if (CG == 2) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = S::TOTAL;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    PB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, p));
    return PB_OK;
  }
  kern<<<grid, kThreads, S::TOTAL, st>>>(p);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// CTA pairs (cta_group::2, gemm.cuh) for the big K-major-A tiles
static bool pair_eligible(const GemmParams& p, int BN, int BK, bool a_mn) {
  // k_iters: a tile with a short K loop (1x1 convolutions on 64..256 channels) is bound by its epilogue / HBM, where the pair
  // only couples two epilogues to one MMA stream
  return BN == 256 && BK == 64 && !a_mn && p.res_iters == 0 && p.a.mode != OP_PATCH_MN && p.b.mode != OP_PATCH_MN &&
         p.k_iters >= 8 && (long long)((p.m_blocks + 1) / 2) * p.n_blocks * p.splits >= num_sms() / 2;
}

// Split-K partial sums are added in a fixed order so that a launch computes the same bits every run (float red.add in
// whatever order the CTAs finish does not).  The slices live in stream-ordered scratch from a memory pool of this library's own
// per device, which keeps what it has allocated (its peak is one step's largest concurrent slices) instead of returning it to
// the driver at every synchronisation; the device's default pool and the framework's allocator are left alone.
int splitk_scratch(float** out, size_t n_floats, cudaStream_t st) {
  constexpr int kMaxDevices = 64;
  static cudaMemPool_t pools[kMaxDevices] = {};
  static std::mutex mu;
  int dev = 0;
  PB_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) return PB_ERR_UNSUPPORTED;
  cudaMemPool_t pool;
  {
    std::lock_guard<std::mutex> lock(mu);
    if (!pools[dev]) {
      cudaMemPoolProps props;
      memset(&props, 0, sizeof(props));
      props.allocType = cudaMemAllocationTypePinned;
      props.location.type = cudaMemLocationTypeDevice;
      props.location.id = dev;
      cudaMemPool_t created;
      PB_CUDA_CHECK(cudaMemPoolCreate(&created, &props));
      uint64_t keep = ~0ull;
      PB_CUDA_CHECK(cudaMemPoolSetAttribute(created, cudaMemPoolAttrReleaseThreshold, &keep));
      pools[dev] = created;
    }
    pool = pools[dev];
  }
  PB_CUDA_CHECK(cudaMallocFromPoolAsync(reinterpret_cast<void**>(out), n_floats * sizeof(float), pool, st));
  return PB_OK;
}

int splitk_release(float* ptr, cudaStream_t st) {
  PB_CUDA_CHECK(cudaFreeAsync(ptr, st));
  return PB_OK;
}

// out[r * ld + c] += part[0][...] + part[1][...] + ... (slices `stride` floats apart), summed in split order; four columns per
// thread (cols, ld and stride are multiples of 4)
__global__ void splitk_reduce_kernel(float* __restrict__ out, const float* __restrict__ part, unsigned rows, unsigned cols4,
                                     long long ld, long long stride, int splits) {
  const unsigned n = rows * cols4;
  for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const unsigned r = e / cols4;
    const long long off = (long long)r * ld + 4ll * (e - r * cols4);
    float4 s = __ldcs(reinterpret_cast<const float4*>(part + off));
    for (int k = 1; k < splits; ++k) {
      const float4 v = __ldcs(reinterpret_cast<const float4*>(part + k * stride + off));
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    float4* o = reinterpret_cast<float4*>(out + off);
    float4 a = *o;
    a.x += s.x; a.y += s.y; a.z += s.z; a.w += s.w;
    *o = a;
  }
}

static int splitk_reduce(float* out, const float* part, long long rows, long long cols, long long ld, long long stride, int splits,
                         cudaStream_t st) {
  if (cols % 4 || ld % 4 || stride % 4 || rows * cols >= (1ll << 32)) return PB_ERR_UNSUPPORTED;
  const long long n = rows * cols / 4;
  const long long cap = (long long)num_sms() * 8;
  const int grid = (int)((n + 255) / 256 < cap ? (n + 255) / 256 : cap);
  splitk_reduce_kernel<<<grid, 256, 0, st>>>(out, part, (unsigned)rows, (unsigned)(cols / 4), ld, stride, splits);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// Runs launch(partial) with scratch for `splits` slices of rows x ld floats (slice s at partial + s * rows * ld, addressed like
// out), adds the slices into out in split order and releases the scratch, also when the launch fails.
int splitk_run(float* out, long long rows, long long cols, long long ld, int splits, cudaStream_t st,
               const std::function<int(float*)>& launch) {
  float* partial = nullptr;
  int rc = splitk_scratch(&partial, (size_t)splits * rows * ld, st);
  if (rc) return rc;
  rc = launch(partial);
  if (!rc) rc = splitk_reduce(out, partial, rows, cols, ld, rows * ld, splits, st);
  const int rc2 = splitk_release(partial, st);
  return rc ? rc : rc2;
}

static int launch_gemm(const GemmParams& p, int BN, int BK, bool a_mn, bool b_mn, cudaStream_t st, int epi = 0, int cg = 1,
                       bool halo = false, int ew = 8) {
  if (p.atomic_add && p.splits > 1 && !p.partial) {
    if (p.ldc % 4 || p.N % 4) return PB_ERR_UNSUPPORTED;
    return splitk_run(reinterpret_cast<float*>(p.out), p.M, p.N, p.ldc, p.splits, st, [&](float* partial) {
      GemmParams q = p;
      q.partial = partial;
      q.part_stride = (long long)p.M * p.ldc;
      return launch_gemm(q, BN, BK, a_mn, b_mn, st, epi, cg, halo, ew);
    });
  }
  if (ew == 16 && epi == 2 && cg == 1 && BN == 256 && BK == 64 && !a_mn && !b_mn && !halo)   // K-small 1x1 convolutions with statistics
    return launch_gemm_t<256, 64, false, false, 2, 1, false, 16>(p, st);
  if (ew == 16 && epi == 1 && BN == 256 && BK == 64 && !a_mn && !halo) {   // epilogue-bound linear launches (GELU / gates)
    if (cg == 2) return b_mn ? launch_gemm_t<256, 64, false, true, 1, 2, false, 16>(p, st) : launch_gemm_t<256, 64, false, false, 1, 2, false, 16>(p, st);
    return b_mn ? launch_gemm_t<256, 64, false, true, 1, 1, false, 16>(p, st) : launch_gemm_t<256, 64, false, false, 1, 1, false, 16>(p, st);
  }
  if (halo && epi >= 1) {      // halo tiles whose 4 x 8 pixel boxes leave through 4-D TMA stores (no residual / gate operand)
    if (BK != 64 || a_mn || b_mn) return PB_ERR_UNSUPPORTED;
    if (BN == 64 && cg == 1) return epi == 2 ? launch_gemm_t<64, 64, false, false, 2, 1, true>(p, st) : launch_gemm_t<64, 64, false, false, 1, 1, true>(p, st);
    if (BN == 256 && cg == 1) return epi == 2 ? launch_gemm_t<256, 64, false, false, 2, 1, true>(p, st) : launch_gemm_t<256, 64, false, false, 1, 1, true>(p, st);
    if (BN == 256 && cg == 2) return epi == 2 ? launch_gemm_t<256, 64, false, false, 2, 2, true>(p, st) : launch_gemm_t<256, 64, false, false, 1, 2, true>(p, st);
    return PB_ERR_UNSUPPORTED;
  }
  if (halo) {      // 3x3 stride-1 convolutions with the halo-box A operand (gemm.cuh HALO)
    if (BK != 64 || a_mn || b_mn || epi != 0) return PB_ERR_UNSUPPORTED;
    if (BN == 256) return cg == 2 ? launch_gemm_t<256, 64, false, false, 0, 2, true>(p, st) : launch_gemm_t<256, 64, false, false, 0, 1, true>(p, st);
    if (BN == 128) return launch_gemm_t<128, 64, false, false, 0, 1, true>(p, st);
    if (BN == 64) return launch_gemm_t<64, 64, false, false, 0, 1, true>(p, st);
    return PB_ERR_UNSUPPORTED;
  }
  if (cg == 2 && BN == 256 && BK == 64 && a_mn && b_mn && epi == 0) return launch_gemm_t<256, 64, true, true, 0, 2>(p, st);
  if (cg == 2 && BN == 256 && BK == 64 && !a_mn) {
    if (epi == 2 && !b_mn) return launch_gemm_t<256, 64, false, false, 2, 2>(p, st);
    if (epi == 1) return b_mn ? launch_gemm_t<256, 64, false, true, 1, 2>(p, st) : launch_gemm_t<256, 64, false, false, 1, 2>(p, st);
    return b_mn ? launch_gemm_t<256, 64, false, true, 0, 2>(p, st) : launch_gemm_t<256, 64, false, false, 0, 2>(p, st);
  }
  if (BK == 128) {     // the generic convolution weight gradient (conv_wgrad_impl): BN 64 or 128
    if (BN == 64) return launch_gemm_t<64, 128, true, true>(p, st);
    if (BN == 128) return launch_gemm_t<128, 128, true, true>(p, st);
    return PB_ERR_UNSUPPORTED;
  }
#define PB_DISPATCH(bn)                                                                 \
  if (BN == bn) {                                                                       \
    if (epi == 2 && !a_mn && !b_mn) return launch_gemm_t<bn, 64, false, false, 2>(p, st); \
    if (epi == 1 && !a_mn && !b_mn) return launch_gemm_t<bn, 64, false, false, 1>(p, st); \
    if (epi == 1 && !a_mn && b_mn) return launch_gemm_t<bn, 64, false, true, 1>(p, st);   \
    if (!a_mn && !b_mn) return launch_gemm_t<bn, 64, false, false>(p, st);              \
    if (!a_mn && b_mn) return launch_gemm_t<bn, 64, false, true>(p, st);                \
    if (a_mn && !b_mn) return launch_gemm_t<bn, 64, true, false>(p, st);                \
    return launch_gemm_t<bn, 64, true, true>(p, st);                                    \
  }
  PB_DISPATCH(64)
  PB_DISPATCH(128)
  PB_DISPATCH(256)
#undef PB_DISPATCH
  return PB_ERR_UNSUPPORTED;
}

static int pick_bn(int m_blocks, int N) {
  if (N <= 64) return 64;
  if (N <= 128) return 128;
  long long t256 = (long long)m_blocks * ((N + 255) / 256);
  if (N % 256 == 0 && t256 >= num_sms()) return 256;
  if (N >= 256 && t256 >= 2 * num_sms()) return 256;
  return 128;
}

static int fill_mat_operand(GemmOperand& op, const void* base, bool mn_major, long long rows, long long K,
                            long long ld, int block_rows, int BK) {
  memset(&op, 0, sizeof(op));
  uint64_t dims[2], strides[1];
  uint32_t box[2];
  strides[0] = (uint64_t)ld * 2;
  if (!mn_major) {
    op.mode = OP_MAT_K;
    dims[0] = (uint64_t)K; dims[1] = (uint64_t)rows;
    box[0] = 64; box[1] = (uint32_t)block_rows;
  } else {
    op.mode = OP_MAT_MN;
    dims[0] = (uint64_t)rows; dims[1] = (uint64_t)K;
    box[0] = 64; box[1] = (uint32_t)BK;
  }
  op.tx_bytes = block_rows * BK * 2;
  op.ntaps = 1;
  return make_tmap_bf16(&op.maps[0], base, 2, dims, strides, box);
}

static void set_epilogue(GemmParams& p, void* out, long long ldc, int out_fp32, int atomic_add, const float* bias,
                         const void* residual, int act, float alpha, float* col_sum) {
  p.out = out; p.ldc = ldc; p.out_fp32 = out_fp32; p.atomic_add = atomic_add;
  p.bias = bias; p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
  p.act = act; p.alpha = alpha; p.col_sum = col_sum;
}

// ---- patch geometry ------------------------------------------------------------------------
static void pick_patch(PatchGeom& g, int Nimg, int Ho, int Wo) {
  g.Nimg = Nimg; g.Ho = Ho; g.Wo = Wo;
  g.TW = Wo < 128 ? Wo : 128;
  g.TH = 128 / g.TW; if (g.TH > Ho) g.TH = Ho; if (g.TH < 1) g.TH = 1;
  g.TN = 1;
  if (g.TH == Ho && g.TW == Wo) { g.TN = 128 / (g.TW * g.TH); if (g.TN > Nimg) g.TN = Nimg; if (g.TN < 1) g.TN = 1; }
  g.wb = (Wo + g.TW - 1) / g.TW;
  g.hb = (Ho + g.TH - 1) / g.TH;
  g.nb = (Nimg + g.TN - 1) / g.TN;
}

// 3x3 (or any <= 3x3, stride 1) convolution through ONE halo box per channel chunk (gemm.cuh HALO): 16 x 8 pixel tiles of one image.
static bool conv_halo_ok(int H, int W, int ntaps, const signed char* dh, const signed char* dw, int& dh0, int& dw0) {
  if (H < 12 || W < 8 || ntaps < 2) return false;
  int hmin = 127, hmax = -127, wmin = 127, wmax = -127;
  for (int t = 0; t < ntaps; ++t) {
    hmin = dh[t] < hmin ? dh[t] : hmin; hmax = dh[t] > hmax ? dh[t] : hmax;
    wmin = dw[t] < wmin ? dw[t] : wmin; wmax = dw[t] > wmax ? dw[t] : wmax;
  }
  if (hmax - hmin > 2 || wmax - wmin > 2) return false;
  // the 16 x 8 tile must cover the image about as well as the row-major 128-pixel patches do (28 x 28: 77 % vs 87.5 % -> no)
  PatchGeom g0;
  pick_patch(g0, 1, H, W);
  const double u_old = (double)H * W / ((double)g0.hb * g0.wb * 128.0);
  const double u_halo = (double)H * W / ((double)((H + kHaloTH - 1) / kHaloTH) * ((W + kHaloTW - 1) / kHaloTW) * 128.0);
  if (u_halo < 0.95 * u_old) return false;
  dh0 = hmin; dw0 = wmin;
  return true;
}
// HALO tiles with a TMA-store epilogue: NHWC output as a 4-D tensor map, box {32 ch, 8, 4, 1} (= one warp's 32 accumulator rows).
// Returns the epilogue variant (1 plain, 2 with column statistics) or 0 when the pixel-addressed epilogue has to stay.
static int halo_lean_epi(GemmParams& p, int BN, int cg, void* out, int N, int Ho, int Wo, int C, const void* residual, int act,
                         float* col_sum) {
  if (residual || act > ACT_RELU || (C % 8) || (reinterpret_cast<uintptr_t>(out) & 15)) return 0;
  if (!((BN == 64 && cg == 1) || BN == 256)) return 0;
  uint64_t dims[4] = {(uint64_t)C, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
  uint64_t str[3] = {(uint64_t)C * 2, (uint64_t)Wo * C * 2, (uint64_t)Ho * Wo * C * 2};
  uint32_t box[4] = {32, (uint32_t)kHaloTW, 4, 1};
  if (make_tmap_bf16(&p.out_map, out, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B) != PB_OK) return 0;
  return col_sum ? 2 : 1;
}
static void halo_geom(PatchGeom& g, int Nimg, int Ho, int Wo) {
  g.Nimg = Nimg; g.Ho = Ho; g.Wo = Wo;
  g.TN = 1; g.TH = kHaloTH; g.TW = kHaloTW;
  g.wb = (Wo + g.TW - 1) / g.TW;
  g.hb = (Ho + g.TH - 1) / g.TH;
  g.nb = Nimg;
}
static int fill_halo_map(GemmOperand& op, const void* base, int N, int H, int W, int C) {
  uint32_t box[4] = {64, (uint32_t)kHaloW, (uint32_t)(kHaloTH + 2), 1};
  uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
  uint64_t str[3] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2};
  return make_tmap_bf16(&op.maps[0], base, 4, dims, str, box);
}

static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
static inline int posmod(int a, int b) { int m = a % b; return m < 0 ? m + b : m; }

// 4D tensor maps over an NHWC tensor [N, H, W, C] (bf16). stride 1 -> one map; stride 2 -> 4 parity maps
// viewing x[:, hp::2, wp::2, :].  Box {64, TW, TH, TN}.
static int fill_patch_maps(GemmOperand& op, const void* base, int N, int H, int W, int C, int src_stride,
                           const PatchGeom& g) {
  uint32_t box[4] = {64, (uint32_t)g.TW, (uint32_t)g.TH, (uint32_t)g.TN};
  if (src_stride == 1) {
    uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2};
    return make_tmap_bf16(&op.maps[0], base, 4, dims, str, box);
  }
  if (src_stride != 2 || (H & 1) || (W & 1)) return PB_ERR_UNSUPPORTED;
  for (int hp = 0; hp < 2; ++hp)
    for (int wp = 0; wp < 2; ++wp) {
      const char* b = reinterpret_cast<const char*>(base) + ((long long)hp * W + wp) * C * 2;
      uint64_t dims[4] = {(uint64_t)C, (uint64_t)(W / 2), (uint64_t)(H / 2), (uint64_t)N};
      uint64_t str[3] = {(uint64_t)2 * C * 2, (uint64_t)2 * W * C * 2, (uint64_t)H * W * C * 2};
      int r = make_tmap_bf16(&op.maps[hp * 2 + wp], b, 4, dims, str, box);
      if (r) return r;
    }
  return PB_OK;
}

// One implicit GEMM of a convolution (the forward, or one output-parity class of the data gradient).  Rows: the pixels of an
// (OH / os) x (OW / os) grid per image, stored to NHWC out [N, OH, OW, cols] at (oh0 + os * h, ow0 + os * w).  A: NHWC src
// [N, Hs, Ws, C] through the per-tap shifts the caller left in p.a.dh / dw / map (src_stride 2: parity maps).  B: wmat
// [cols][ntaps * C].  A stride-1 convolution whose output has the extent of its input may take the HALO tiles; with a
// residual only when halo_residual.
static int conv_igemm(GemmParams& p, const void* src, int N, int Hs, int Ws, int C, int src_stride, int ntaps, const void* wmat,
                      int cols, void* out, int OH, int OW, int os, int oh0, int ow0, const float* bias, const void* residual,
                      int act, float* col_sum, bool halo_residual, cudaStream_t st) {
  const int Hg = OH / os, Wg = OW / os;
  const bool halo = src_stride == 1 && os == 1 && OH == Hs && OW == Ws && (halo_residual || !residual) &&
                    conv_halo_ok(Hs, Ws, ntaps, p.a.dh, p.a.dw, p.halo_dh0, p.halo_dw0);
  if (halo) halo_geom(p.geom, N, Hg, Wg);
  else pick_patch(p.geom, N, Hg, Wg);
  p.M = N * Hg * Wg; p.N = cols;
  p.m_blocks = p.geom.nb * p.geom.hb * p.geom.wb;
  const int BN = pick_bn(p.m_blocks, cols);
  p.n_blocks = (cols + BN - 1) / BN;
  p.splits = 1;
  p.a.mode = OP_PATCH_K;
  p.a.cchunks = C / 64;
  p.a.ntaps = ntaps;
  p.a.tx_bytes = p.geom.TN * p.geom.TH * p.geom.TW * 128;
  int rc = halo ? fill_halo_map(p.a, src, N, Hs, Ws, C) : fill_patch_maps(p.a, src, N, Hs, Ws, C, src_stride, p.geom);
  if (rc) return rc;
  p.k_iters = ntaps * p.a.cchunks;
  p.k_steps = 4;
  // (CTA pairs on the 64-wide halo tiles were measured and dropped: 64 ch at 56x56 forward 453 -> 545 us, dgrad 427 -> 501 us)
  const int cg = pair_eligible(p, BN, 64, false) ? 2 : 1;
  rc = fill_mat_operand(p.b, wmat, false, cols, (long long)ntaps * C, (long long)ntaps * C, BN / cg, 64);
  if (rc) return rc;
  set_epilogue(p, out, cols, 0, 0, bias, residual, act, 1.f, col_sum);
  p.out_pixel = 1; p.OH = OH; p.OW = OW; p.osh = os; p.osw = os; p.oh0 = oh0; p.ow0 = ow0;
  const int hepi = halo ? halo_lean_epi(p, BN, cg, out, N, OH, OW, cols, residual, act, col_sum) : 0;
  return launch_gemm(p, BN, 64, false, false, st, hepi, cg, halo);
}

}  // namespace pb

using namespace pb;

// ==============================================================================================
// Dense GEMM
// ==============================================================================================
extern "C" int passl_b200_gemm_bf16(const void* A, const void* B, void* out, int M, int N, int K, int a_mn_major,
                                    int b_mn_major, long long lda, long long ldb, long long ldc, int out_fp32,
                                    int atomic_add, const float* bias, const void* residual, int act, float alpha,
                                    int splits, float* col_sum, float* col_sqsum, void* stream) {
  return passl_b200_gemm_bf16_ex(A, B, out, M, N, K, a_mn_major, b_mn_major, lda, ldb, ldc, out_fp32, atomic_add, bias,
                                 residual, act, alpha, splits, col_sum, col_sqsum, nullptr, 0, nullptr, stream);
}

extern "C" int passl_b200_gemm_bf16_ex(const void* A, const void* B, void* out, int M, int N, int K, int a_mn_major,
                                       int b_mn_major, long long lda, long long ldb, long long ldc, int out_fp32,
                                       int atomic_add, const float* bias, const void* residual, int act, float alpha,
                                       int splits, float* col_sum, float* col_sqsum, const void* aux, int aux_mode,
                                       void* preact_out, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return PB_ERR_BAD_ARG;
  if ((lda % 8) || (ldb % 8) || (N % 8) || (ldc % (out_fp32 ? 4 : 8))) return PB_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(out)) & 15) return PB_ERR_BAD_ARG;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N;
  p.m_blocks = (M + 127) / 128;
  int BN = pick_bn(p.m_blocks, N);
  p.n_blocks = (N + BN - 1) / BN;
  p.k_iters = (K + 63) / 64;
  p.k_steps = 4;
  if (splits < 1) splits = 1;
  if (splits > p.k_iters) splits = p.k_iters;
  if (splits > 1 && !(out_fp32 && atomic_add)) return PB_ERR_BAD_ARG;
  // Weight gradients of the linear layers (both operands MN-major, fp32 split-K accumulation): 128 x 128 tiles pull 256 B/clk/SM
  // from L2 at full MMA rate (delivered: ~50), so they ran at 0.45-0.65 of a plain GEMM.  A CTA pair on a 256 x 256 tile needs half
  // of that per SM; the caller's split count is replaced by the one that minimises whole waves of num_sms / 2 clusters x item length.
  bool wgrad_pair = false;
  if (a_mn_major && b_mn_major && out_fp32 && atomic_add && splits > 1 && N % 256 == 0 && M >= 256 && !bias && !residual && !aux) {
    const int slots = num_sms() / 2;
    const int ptiles = ((p.m_blocks + 1) / 2) * (N / 256);
    // cost of a split count in K iterations: whole waves x (iterations per item + ~32 for the pipeline fill and the 128 KB of
    // fp32 reductions each CTA issues per item)
    int best = 0; long long best_cost = 0;
    const int smax = p.k_iters / 16 < 64 ? p.k_iters / 16 : 64;
    for (int sp = 1; sp <= smax; ++sp) {
      const long long items = (long long)ptiles * sp;
      const long long waves = (items + slots - 1) / slots;
      const long long cost = waves * ((p.k_iters + sp - 1) / sp + 32);
      if (best == 0 || cost < best_cost) { best_cost = cost; best = sp; }
    }
    if (best > 0) { BN = 256; p.n_blocks = N / 256; splits = best; wgrad_pair = true; }
  }
  p.splits = splits;
  int r = fill_mat_operand(p.a, A, a_mn_major != 0, M, K, lda, 128, 64);
  if (r) return r;
  // CTA pairs: each CTA loads half of the B tile (its own box of BN / 2 rows); the residual then enters through the epilogue
  // not for epilogue-bound launches (GELU / gate arithmetic: the pair couples two epilogues to one MMA stream, measured 5 % slower),
  // nor when a residual could ride the MMA of a short K loop instead of the epilogue (proj of ViT-B: 999 vs 917 TF/s)
  // GELU / gate launches: epilogue-bound.  With 8 epilogue warps a pair only couples two slow epilogues to one MMA stream (-5 %);
  // with 16 warps per CTA and K >= 768 the pair wins (fc2-dgrad + GELU' 817 -> 1011 TF/s, fc1 + GELU 1017 -> 1064 at the CLIP batch;
  // K = 512: 798 -> 753, so those stay single).
  const bool heavy = act == ACT_GELU || act == ACT_QUICKGELU || (aux && aux_mode >= 2);
  const bool heavy_pair_ok = heavy && K >= 768;
  const bool heavy_epi = heavy && !heavy_pair_ok;
  const bool short_k_residual = residual && K < 1536;
  const int cg = (wgrad_pair || (!heavy_epi && !short_k_residual && pair_eligible(p, BN, 64, a_mn_major != 0))) ? 2 : 1;
  r = fill_mat_operand(p.b, B, b_mn_major != 0, N, K, ldb, BN / cg, 64);
  if (r) return r;
  set_epilogue(p, out, ldc, out_fp32, atomic_add, bias, residual, act, alpha, col_sum);
  p.aux = reinterpret_cast<const __nv_bfloat16*>(aux);
  p.aux_mode = aux_mode;
  p.preact = reinterpret_cast<__nv_bfloat16*>(preact_out);
  if (cg == 1) {
    r = setup_residual_mma(p, residual, ldc, (cudaStream_t)stream);
    if (r) return r;
  }
  // linear-layer epilogue (EPI 1, TMA stores): plain row-major bf16 output, K-major A, no statistics / scaling, at most one
  // operand tile (gate operand or a residual that does not go through the MMA)
  int epi = 0;
  const bool res_in_epilogue = residual && p.res_iters == 0;
  const bool stats_ok = !col_sum || (!b_mn_major && act <= ACT_RELU && !preact_out && (!aux || aux_mode == 1));   // EPI 2
  if (!out_fp32 && !a_mn_major && stats_ok && alpha == 1.f && splits == 1 && !(aux && res_in_epilogue) &&
      !((reinterpret_cast<uintptr_t>(aux) | reinterpret_cast<uintptr_t>(preact_out) | reinterpret_cast<uintptr_t>(residual)) & 15)) {
    uint64_t dims[2] = {(uint64_t)N, (uint64_t)M}, strides[1] = {(uint64_t)ldc * 2};
    uint32_t box[2] = {32, 32};
    r = make_tmap_bf16(&p.out_map, out, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
    if (r) return r;
    if (preact_out) {
      r = make_tmap_bf16(&p.pre_map, preact_out, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
      if (r) return r;
    }
    const void* tsrc = aux ? aux : (res_in_epilogue ? residual : nullptr);
    if (tsrc) {
      uint32_t tbox[2] = {(uint32_t)(BN < N ? BN : N), 128};
      if (tbox[0] <= 256 && make_tmap_bf16(&p.tile_map, tsrc, 2, dims, strides, tbox, CU_TENSOR_MAP_SWIZZLE_NONE) == PB_OK) p.tile_prefetch = 1;
    }
    epi = col_sum ? 2 : 1;
  }
  // 16 epilogue warps (3 pipeline stages, accumulator read in place): fc2-dgrad with the GELU' gate 647 -> 801 TF/s at the CLIP
  // batch, 597 -> 760 at the MAE decoder's; fc1 forward (+GELU, saved pre-activation) gains only with a short K loop (K = 512:
  // 746 -> 783, K = 768: 940 -> 917), `profiles/r02_vit_gemm_probe_ew16.txt`
  // (also the 1x1 convolutions with BatchNorm statistics and a K loop of <= 4 iterations: one MMA group per tile, the epilogue is all
  // there is)
  const bool use16 = (aux && aux_mode >= 2) || ((act == ACT_GELU || act == ACT_QUICKGELU) && (K < 768 || (heavy_pair_ok && cg == 2))) ||
                     (epi == 2 && cg == 1 && p.k_iters <= 4);
  return launch_gemm(p, BN, 64, a_mn_major != 0, b_mn_major != 0, (cudaStream_t)stream, epi, cg, false, use16 ? 16 : 8);
}

extern "C" int passl_b200_gemm_stats_rows(void) { return 4 * num_sms(); }

// ==============================================================================================
// Convolution forward (implicit GEMM), NHWC bf16, weights [Cout, R, S, Cin] bf16.
//   out[n, p, q, co] = epilogue( sum_{r,s,ci} x[n, p*stride + r - pad, q*stride + s - pad, ci] * w[co, r, s, ci] )
// ==============================================================================================
static int conv_fwd_impl(const void* x, const void* w, void* out, int N, int H, int W, int Cin, int Cout, int R, int S,
                         int stride, int pad_h, int pad_w, int Ho, int Wo, const float* bias, const void* residual, int act,
                         float* col_sum, void* stream) {
  if (Cin % 64 || Cout % 8 || R * S > kMaxTaps) return PB_ERR_UNSUPPORTED;
  if (R == 1 && S == 1 && stride == 1 && pad_h == 0 && pad_w == 0 && Ho == H && Wo == W) {
    return passl_b200_gemm_bf16(x, w, out, N * H * W, Cout, Cin, 0, 0, Cin, Cin, Cout, 0, 0, bias, residual, act,
                                1.f, 1, col_sum, nullptr, stream);
  }
  GemmParams p;
  memset(&p, 0, sizeof(p));
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < S; ++s) {
      int t = r * S + s;
      int th = r - pad_h, tw = s - pad_w;
      p.a.dh[t] = (signed char)floordiv(th, stride);
      p.a.dw[t] = (signed char)floordiv(tw, stride);
      p.a.map[t] = (signed char)(stride == 1 ? 0 : posmod(th, 2) * 2 + posmod(tw, 2));
    }
  return conv_igemm(p, x, N, H, W, Cin, stride, R * S, w, Cout, out, Ho, Wo, 1, 0, 0, bias, residual, act, col_sum, false,
                    (cudaStream_t)stream);
}

extern "C" int passl_b200_conv2d_fwd_bf16(const void* x, const void* w, void* out, int N, int H, int W, int Cin,
                                          int Cout, int R, int S, int stride, int pad, const float* bias,
                                          const void* residual, int act, float* col_sum, float* col_sqsum,
                                          void* stream) {
  const int Ho = (H + 2 * pad - R) / stride + 1, Wo = (W + 2 * pad - S) / stride + 1;
  return conv_fwd_impl(x, w, out, N, H, W, Cin, Cout, R, S, stride, pad, pad, Ho, Wo, bias, residual, act, col_sum, stream);
}

// Rectangular filters with separate row / column padding and an explicit output extent (stride 1): the W-unfolded
// space-to-depth form of the 7x7/2 stem is a 4x1 convolution over 64 channels with rows padded (2, 1).
extern "C" int passl_b200_conv2d_fwd_rect_bf16(const void* x, const void* w, void* out, int N, int H, int W, int Cin,
                                               int Cout, int R, int S, int pad_h, int pad_w, int Ho, int Wo,
                                               const float* bias, int act, float* col_sum, void* stream) {
  if (Ho <= 0 || Wo <= 0 || Ho > H + 2 * pad_h - R + 1 + R || Wo > W + 2 * pad_w - S + 1 + S) return PB_ERR_BAD_ARG;
  return conv_fwd_impl(x, w, out, N, H, W, Cin, Cout, R, S, 1, pad_h, pad_w, Ho, Wo, bias, nullptr, act, col_sum, stream);
}

// ==============================================================================================
// Convolution data gradient.  dx[n,h,w,ci] = sum dy[n,p,q,co] * w[co,r,s,ci]  over (p,q,r,s) with
// h = p*stride + r - pad.  Runs one implicit GEMM per output-parity class over dy with class weights
// wt[class][ci][tap][co] gathered by passl_b200_conv2d_dgrad_prepare_weights (same call order).
//   accumulate != 0 : dx += result (dx already holds another branch's gradient), else dx = result.
// ==============================================================================================
namespace pb {
struct DgradClass {
  int a, b, ntaps;
  int r[kMaxTaps], s[kMaxTaps], dh[kMaxTaps], dw[kMaxTaps];
};
static int build_dgrad_classes(DgradClass* cls, int R, int S, int stride, int pad) {
  int n = 0;
  for (int a = 0; a < stride; ++a)
    for (int b = 0; b < stride; ++b) {
      DgradClass& c = cls[n++];
      c.a = a; c.b = b; c.ntaps = 0;
      for (int r = 0; r < R; ++r) {
        if (posmod(a + pad - r, stride)) continue;
        for (int s = 0; s < S; ++s) {
          if (posmod(b + pad - s, stride)) continue;
          int t = c.ntaps++;
          c.r[t] = r; c.s[t] = s;
          c.dh[t] = floordiv(a + pad - r, stride);
          c.dw[t] = floordiv(b + pad - s, stride);
        }
      }
    }
  return n;
}

__global__ void weight_gather_kernel(const __nv_bfloat16* __restrict__ w, __nv_bfloat16* __restrict__ wt, int Cout,
                                     int Cin, int R, int S, int ntaps, const int4 taps_rs_lo, const int4 taps_rs_hi,
                                     const int4 taps_rs_top) {
  // wt[ci][t][co] = w[co][r_t][s_t][ci];  taps packed as r*16+s in 12 ints
  int packed[12] = {taps_rs_lo.x, taps_rs_lo.y, taps_rs_lo.z, taps_rs_lo.w, taps_rs_hi.x, taps_rs_hi.y,
                    taps_rs_hi.z, taps_rs_hi.w, taps_rs_top.x, taps_rs_top.y, taps_rs_top.z, taps_rs_top.w};
  __shared__ __nv_bfloat16 tile[32][33];
  int t = blockIdx.z;
  int r = packed[t] >> 4, s = packed[t] & 15;
  int co0 = blockIdx.y * 32, ci0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int co = co0 + i, ci = ci0 + threadIdx.x;
    if (co < Cout && ci < Cin) tile[i][threadIdx.x] = w[(((long long)co * R + r) * S + s) * Cin + ci];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int ci = ci0 + i, co = co0 + threadIdx.x;
    if (co < Cout && ci < Cin) wt[((long long)ci * ntaps + t) * Cout + co] = tile[threadIdx.x][i];
  }
}
}  // namespace pb

extern "C" long long passl_b200_conv2d_dgrad_workspace_bytes(int Cin, int Cout, int R, int S) {
  return (long long)Cin * Cout * R * S * 2 + 1024;
}

extern "C" int passl_b200_conv2d_dgrad_bf16(const void* dy, const void* w, void* dx, void* workspace, int N, int H,
                                            int W, int Cin, int Cout, int R, int S, int stride, int pad,
                                            int accumulate, void* stream) {
  if (Cout % 64 || Cin % 8 || R * S > kMaxTaps || (stride != 1 && stride != 2)) return PB_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int Ho = (H + 2 * pad - R) / stride + 1, Wo = (W + 2 * pad - S) / stride + 1;
  if (R == 1 && S == 1 && stride == 1 && pad == 0) {
    // dx[P, Cin] = dy[P, Cout] * w[Cout, Cin]  (B is MN-major: no weight transform)
    return passl_b200_gemm_bf16(dy, w, dx, N * H * W, Cin, Cout, 0, 1, Cout, Cin, Cin, 0, 0, nullptr,
                                accumulate ? dx : nullptr, ACT_NONE, 1.f, 1, nullptr, nullptr, stream);
  }
  if (stride == 2 && ((H & 1) || (W & 1))) return PB_ERR_UNSUPPORTED;
  DgradClass cls[4];
  int ncls = build_dgrad_classes(cls, R, S, stride, pad);
  bool any_empty = false;
  for (int c = 0; c < ncls; ++c) any_empty |= (cls[c].ntaps == 0);
  if (any_empty && !accumulate) PB_CUDA_CHECK(cudaMemsetAsync(dx, 0, (size_t)N * H * W * Cin * 2, st));
  __nv_bfloat16* wt = reinterpret_cast<__nv_bfloat16*>(workspace);
  for (int c = 0; c < ncls; ++c) {
    const DgradClass& k = cls[c];
    if (k.ntaps == 0) continue;
    int packed[12] = {0};
    for (int t = 0; t < k.ntaps; ++t) packed[t] = k.r[t] * 16 + k.s[t];
    dim3 grid((Cin + 31) / 32, (Cout + 31) / 32, k.ntaps), block(32, 8);
    weight_gather_kernel<<<grid, block, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(w), wt, Cout, Cin, R, S,
                                                 k.ntaps, make_int4(packed[0], packed[1], packed[2], packed[3]),
                                                 make_int4(packed[4], packed[5], packed[6], packed[7]),
                                                 make_int4(packed[8], packed[9], packed[10], packed[11]));
    PB_LAUNCH_CHECK();
    GemmParams p;
    memset(&p, 0, sizeof(p));
    for (int t = 0; t < k.ntaps; ++t) { p.a.dh[t] = (signed char)k.dh[t]; p.a.dw[t] = (signed char)k.dw[t]; }
    const int rc = conv_igemm(p, dy, N, Ho, Wo, Cout, 1, k.ntaps, wt, Cin, dx, H, W, stride, k.a, k.b, nullptr,
                              accumulate ? dx : nullptr, ACT_NONE, nullptr, true, st);
    if (rc) return rc;
    wt += (size_t)Cin * k.ntaps * Cout;
  }
  return PB_OK;
}

// ==============================================================================================
// Convolution weight gradient: dw[co, r, s, ci] (fp32, atomically accumulated) =
//     sum_{n,p,q} dy[n,p,q,co] * x[n, p*stride + r - pad, q*stride + s - pad, ci]
// K = output pixels (patch tiles), split across CTAs.
// ==============================================================================================
namespace pb {
int launch_wgrad_halo(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin, int Cout, int R, int S, int pad_h,
                      int pad_w, cudaStream_t st);
}

static int conv_wgrad_impl(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin, int Cout, int R, int S,
                           int stride, int pad_h, int pad_w, int Ho, int Wo, int zero_first, void* stream) {
  if (Cin % 8 || Cout % 8 || R * S > kMaxTaps || (stride != 1 && stride != 2)) return PB_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int pad = pad_h;
  if (zero_first) PB_CUDA_CHECK(cudaMemsetAsync(dw, 0, (size_t)Cout * R * S * Cin * 4, st));
  if (R == 1 && S == 1 && stride == 1 && pad_h == 0 && pad_w == 0 && Ho == H && Wo == W) {
    int P = N * H * W;
    int mb = (Cout + 127) / 128;
    int BNg = pick_bn(mb, Cin);
    int tiles = mb * ((Cin + BNg - 1) / BNg);
    int splits = (2 * num_sms() + tiles - 1) / tiles;
    int kit = (P + 63) / 64;
    if (splits > kit / 4) splits = kit / 4 > 0 ? kit / 4 : 1;
    return passl_b200_gemm_bf16(dy, x, dw, Cout, Cin, P, 1, 1, Cout, Cin, Cin, 1, 1, nullptr, nullptr, ACT_NONE, 1.f,
                                splits, nullptr, nullptr, stream);
  }
  if (stride == 1 && Ho == H && Wo == W && R * S > 1) {
    // halo-tile kernel (wgrad_halo.cu): one TMA halo load serves all taps; falls through when the shape is outside its contract
    int rc = launch_wgrad_halo(x, dy, dw, N, H, W, Cin, Cout, R, S, pad_h, pad_w, st);
    if (rc != PB_ERR_UNSUPPORTED) return rc;
  }
  GemmParams p;
  memset(&p, 0, sizeof(p));
  pick_patch(p.geom, N, Ho, Wo);
  const int rows = p.geom.TN * p.geom.TH * p.geom.TW;
  p.M = Cout; p.N = R * S * Cin;
  p.m_blocks = (Cout + 127) / 128;
  int BN = Cin <= 64 ? 64 : 128;
  p.n_blocks_per_tap = (Cin + BN - 1) / BN;
  p.n_per_tap = Cin;
  p.n_blocks = R * S * p.n_blocks_per_tap;
  p.k_iters = p.geom.nb * p.geom.hb * p.geom.wb;
  p.k_steps = (rows + 15) / 16;
  int tiles = p.m_blocks * p.n_blocks;
  int splits = (2 * num_sms() + tiles - 1) / tiles;
  if (splits > p.k_iters) splits = p.k_iters;
  if (splits < 1) splits = 1;
  p.splits = splits;
  // A = dy patches (channels = M rows), B = x patches shifted by the tap (channels = N rows)
  p.a.mode = OP_PATCH_MN; p.a.ntaps = 1; p.a.tx_bytes = 2 * rows * 128;
  p.a.dh[0] = 0; p.a.dw[0] = 0; p.a.map[0] = 0;
  int rc = fill_patch_maps(p.a, dy, N, Ho, Wo, Cout, 1, p.geom);
  if (rc) return rc;
  p.b.mode = OP_PATCH_MN; p.b.ntaps = R * S; p.b.tx_bytes = (BN / 64) * rows * 128;
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < S; ++s) {
      int t = r * S + s;
      int th = r - pad, tw = s - pad_w;
      p.b.dh[t] = (signed char)floordiv(th, stride);
      p.b.dw[t] = (signed char)floordiv(tw, stride);
      p.b.map[t] = (signed char)(stride == 1 ? 0 : posmod(th, 2) * 2 + posmod(tw, 2));
    }
  rc = fill_patch_maps(p.b, x, N, H, W, Cin, stride, p.geom);
  if (rc) return rc;
  set_epilogue(p, dw, (long long)R * S * Cin, 1, 1, nullptr, nullptr, ACT_NONE, 1.f, nullptr);
  return launch_gemm(p, BN, 128, true, true, st);
}

extern "C" int passl_b200_conv2d_wgrad_bf16(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin,
                                            int Cout, int R, int S, int stride, int pad, int zero_first,
                                            void* stream) {
  const int Ho = (H + 2 * pad - R) / stride + 1, Wo = (W + 2 * pad - S) / stride + 1;
  return conv_wgrad_impl(x, dy, dw, N, H, W, Cin, Cout, R, S, stride, pad, pad, Ho, Wo, zero_first, stream);
}

extern "C" int passl_b200_conv2d_wgrad_rect_bf16(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin,
                                                 int Cout, int R, int S, int pad_h, int pad_w, int Ho, int Wo, int zero_first,
                                                 void* stream) {
  if (Ho <= 0 || Wo <= 0) return PB_ERR_BAD_ARG;
  return conv_wgrad_impl(x, dy, dw, N, H, W, Cin, Cout, R, S, 1, pad_h, pad_w, Ho, Wo, zero_first, stream);
}
