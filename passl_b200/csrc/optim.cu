// Fused optimizer steps over flat fp32 parameter / gradient buffers (SURVEY.md §8 f-1: the step right after the path).
// One launch updates every parameter of a group and refreshes the bf16 compute copy the tcgen05 kernels read.
//
// Reference semantics:
//   Momentum  (passl/optimizer/momentum.py:60-158, paddle Momentum w/ L2Decay):  g' = g + wd*p; v = mu*v + g'; p -= lr*v
//   LARS      (passl/optimizer/momentum_lars.py:56-114, paddle LarsMomentum):    local_lr = lr*coeff*||p||/(||g|| + wd*||p|| + eps)
//                                                                               v = mu*v + local_lr*(g + wd*p); p -= v
//   AdamW     (passl/optimizer/adamw.py:52-138 -> _C_ops.adamw):  decoupled decay p *= (1 - lr*wd), bias-corrected Adam
// Parameters live in a flat buffer whose tensors start at multiples of 1024 elements (ParamStore), so a 1024-element
// block never straddles two tensors: `block_seg[b]` gives the tensor id of block b for the per-tensor LARS norms.
#include "common.cuh"
#include "host_utils.h"
#include "../../include/passl_b200.h"

namespace pb {

int splitk_scratch(float** out, size_t n_floats, cudaStream_t st);     // gemm_api.cu: stream-ordered scratch
int splitk_release(float* ptr, cudaStream_t st);

constexpr int OPT_BLOCK = 1024;  // elements per CTA (256 threads x 4)

__device__ __forceinline__ void store_bf16x4(__nv_bfloat16* dst, const float4& v) {
  uint2 u;
  u.x = pack_bf16x2(v.x, v.y);
  u.y = pack_bf16x2(v.z, v.w);
  *reinterpret_cast<uint2*>(dst) = u;
}

__global__ void sgd_momentum_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ v,
                                    __nv_bfloat16* __restrict__ p_bf16, float lr, float mu, float wd, float gscale,
                                    const float* __restrict__ ctrl, long long n) {
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  if (ctrl) {                      // {multiplier, found_inf, global norm} written by grad_norm_finite_kernel
    if (ctrl[1] != 0.f) return;    // non-finite gradient: the step is skipped (grad_scaler.py:48-87)
    gscale *= ctrl[0];
  }
  float4 pp = *reinterpret_cast<float4*>(p + i), gg = *reinterpret_cast<const float4*>(g + i), vv = *reinterpret_cast<float4*>(v + i);
  vv.x = mu * vv.x + (gg.x * gscale + wd * pp.x); pp.x -= lr * vv.x;
  vv.y = mu * vv.y + (gg.y * gscale + wd * pp.y); pp.y -= lr * vv.y;
  vv.z = mu * vv.z + (gg.z * gscale + wd * pp.z); pp.z -= lr * vv.z;
  vv.w = mu * vv.w + (gg.w * gscale + wd * pp.w); pp.w -= lr * vv.w;
  *reinterpret_cast<float4*>(p + i) = pp;
  *reinterpret_cast<float4*>(v + i) = vv;
  if (p_bf16) store_bf16x4(p_bf16 + i, pp);
}

// per-block squared norms: part[2*block] = sum p^2, part[2*block+1] = sum (g*gscale)^2 (seg_norm_finalize_kernel adds them per tensor)
__global__ void seg_sqnorm_kernel(const float* __restrict__ p, const float* __restrict__ g, float* __restrict__ part, float gscale,
                                  long long n) {
  __shared__ float red[2][8];
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  float a = 0.f, b = 0.f;
  if (i < n) {
    float4 pp = *reinterpret_cast<const float4*>(p + i), gg = *reinterpret_cast<const float4*>(g + i);
    a = pp.x * pp.x + pp.y * pp.y + pp.z * pp.z + pp.w * pp.w;
    gg.x *= gscale; gg.y *= gscale; gg.z *= gscale; gg.w *= gscale;
    b = gg.x * gg.x + gg.y * gg.y + gg.z * gg.z + gg.w * gg.w;
  }
  a = warp_sum(a); b = warp_sum(b);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[0][w] = a; red[1][w] = b; }
  __syncthreads();
  if (w == 0) {
    a = l < 8 ? red[0][l] : 0.f; b = l < 8 ? red[1][l] : 0.f;
    a = warp_sum(a); b = warp_sum(b);
    if (l == 0) {
      part[2 * blockIdx.x] = a;
      part[2 * blockIdx.x + 1] = b;
    }
  }
}

// one CTA per tensor: norms[2*seg + {0,1}] = the sums of that tensor's block partials in a fixed order, so the LARS trust ratio
// is the same every run (block_seg is non-decreasing: a tensor's blocks are contiguous)
__global__ void seg_norm_finalize_kernel(const float* __restrict__ part, const int* __restrict__ block_seg, int nblocks,
                                         float* __restrict__ norms) {
  __shared__ float red[2][8];
  const int s = blockIdx.x;
  int lo = 0, hi = nblocks;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (block_seg[mid] < s) lo = mid + 1; else hi = mid; }
  const int b0 = lo;
  hi = nblocks;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (block_seg[mid] <= s) lo = mid + 1; else hi = mid; }
  float a = 0.f, b = 0.f;
  for (int k = b0 + (int)threadIdx.x; k < lo; k += blockDim.x) { a += part[2 * k]; b += part[2 * k + 1]; }
  a = warp_sum(a); b = warp_sum(b);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[0][w] = a; red[1][w] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ta = 0.f, tb = 0.f;
    for (int k = 0; k < 8; ++k) { ta += red[0][k]; tb += red[1][k]; }
    norms[2 * s] = ta;
    norms[2 * s + 1] = tb;
  }
}

__global__ void lars_momentum_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ v,
                                     __nv_bfloat16* __restrict__ p_bf16, const int* __restrict__ block_seg,
                                     const float* __restrict__ norms, const float* __restrict__ seg_wd, float lr, float mu,
                                     float coeff, float eps, float gscale, const float* __restrict__ ctrl, long long n) {
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  float cm = 1.f;
  if (ctrl) {
    if (ctrl[1] != 0.f) return;
    cm = ctrl[0];
    gscale *= cm;
  }
  const int s = block_seg[blockIdx.x];
  const float wd = seg_wd[s];
  const float pn = sqrtf(norms[2 * s]), gn = sqrtf(norms[2 * s + 1]) * cm;   // the norms were taken before the clip multiplier
  float local_lr = lr;
  if (wd > 0.f && pn > 0.f && gn > 0.f) local_lr = lr * coeff * pn / (gn + wd * pn + eps);
  float4 pp = *reinterpret_cast<float4*>(p + i), gg = *reinterpret_cast<const float4*>(g + i), vv = *reinterpret_cast<float4*>(v + i);
  vv.x = mu * vv.x + local_lr * (gg.x * gscale + wd * pp.x); pp.x -= vv.x;
  vv.y = mu * vv.y + local_lr * (gg.y * gscale + wd * pp.y); pp.y -= vv.y;
  vv.z = mu * vv.z + local_lr * (gg.z * gscale + wd * pp.z); pp.z -= vv.z;
  vv.w = mu * vv.w + local_lr * (gg.w * gscale + wd * pp.w); pp.w -= vv.w;
  *reinterpret_cast<float4*>(p + i) = pp;
  *reinterpret_cast<float4*>(v + i) = vv;
  if (p_bf16) store_bf16x4(p_bf16 + i, pp);
}

__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                             __nv_bfloat16* __restrict__ p_bf16, const int* __restrict__ block_seg,
                             const float* __restrict__ seg_wd, const float* __restrict__ seg_lr_ratio, float lr, float b1,
                             float b2, float eps, float bc1, float bc2, float gscale, const float* __restrict__ ctrl,
                             long long n) {
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  if (ctrl) {
    if (ctrl[1] != 0.f) return;
    gscale *= ctrl[0];
  }
  const int s = block_seg ? block_seg[blockIdx.x] : 0;
  const float wd = seg_wd ? seg_wd[s] : 0.f;
  const float lrs = lr * (seg_lr_ratio ? seg_lr_ratio[s] : 1.f);
  float4 pp = *reinterpret_cast<float4*>(p + i), gg = *reinterpret_cast<const float4*>(g + i);
  float4 mm = *reinterpret_cast<float4*>(m + i), vv = *reinterpret_cast<float4*>(v + i);
  float* P = reinterpret_cast<float*>(&pp); float* G = reinterpret_cast<float*>(&gg);
  float* M = reinterpret_cast<float*>(&mm); float* V = reinterpret_cast<float*>(&vv);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float gj = G[j] * gscale;
    P[j] *= (1.f - lrs * wd);
    M[j] = b1 * M[j] + (1.f - b1) * gj;
    V[j] = b2 * V[j] + (1.f - b2) * gj * gj;
    float mh = M[j] / bc1, vh = V[j] / bc2;
    P[j] -= lrs * mh / (sqrtf(vh) + eps);
  }
  *reinterpret_cast<float4*>(p + i) = pp;
  *reinterpret_cast<float4*>(m + i) = mm;
  *reinterpret_cast<float4*>(v + i) = vv;
  if (p_bf16) store_bf16x4(p_bf16 + i, pp);
}

// One pass over the flat gradient buffer: sum of squares + non-finite flag; the last CTA turns them into the control word the
// optimizer kernels read:  ctrl = {multiplier, found_inf, global_norm}
//   multiplier = unscale * clip_coef,  clip_coef = 1 if (!always_clip && norm <= clip_norm) else min(clip_norm / (norm + 1e-6), coef_max)
// (passl/core/grad_clip.py:30-84 ClipGradByGlobalNorm; passl/core/grad_scaler.py:48-87 check_finite_and_unscale).  `unscale` folds
// 1/loss_scale and the 1/world of the gradient mean.  scratch: {sumsq, found, ticket} zeroed once, left zeroed.
__global__ void grad_norm_finite_kernel(const float* __restrict__ g, long long n, float unscale, float clip_norm, float coef_max,
                                        int always_clip, float* __restrict__ ctrl, float* __restrict__ scratch) {
  __shared__ float red[8];
  __shared__ int red_bad[8];
  float a = 0.f;
  int bad = 0;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += (long long)gridDim.x * blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4*>(g + i);
    a += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    bad |= !(fabsf(v.x) <= 3.4e38f) | !(fabsf(v.y) <= 3.4e38f) | !(fabsf(v.z) <= 3.4e38f) | !(fabsf(v.w) <= 3.4e38f);
  }
  a = warp_sum(a);
  bad = __any_sync(0xffffffffu, bad);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[w] = a; red_bad[w] = bad; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    int b = 0;
    for (int k = 0; k < 8; ++k) { t += red[k]; b |= red_bad[k]; }
    atomicAdd(scratch, t);
    if (b) atomicExch(reinterpret_cast<unsigned*>(scratch + 1), 1u);
    __threadfence();
    unsigned* ticket = reinterpret_cast<unsigned*>(scratch + 2);
    if (atomicInc(ticket, gridDim.x - 1) == gridDim.x - 1) {
      __threadfence();
      const float sumsq = __ldcg(scratch);
      const unsigned found = __ldcg(reinterpret_cast<unsigned*>(scratch + 1));
      const float norm = sqrtf(sumsq) * fabsf(unscale);
      float coef = 1.f;
      if (clip_norm > 0.f && (always_clip || norm > clip_norm)) {
        coef = clip_norm / (norm + 1e-6f);
        if (coef_max > 0.f) coef = fminf(coef, coef_max);
      }
      const bool inf = found != 0u || !(sumsq <= 3.4e38f);
      ctrl[0] = inf ? 0.f : unscale * coef;
      ctrl[1] = inf ? 1.f : 0.f;
      ctrl[2] = norm;
      scratch[0] = 0.f;
      *reinterpret_cast<unsigned*>(scratch + 1) = 0u;
    }
  }
}

}  // namespace pb

using namespace pb;

// ctrl fp32[3] (output), scratch fp32[3] (zeroed once by the caller).  clip_norm <= 0: no clipping (finite check + unscale only).
extern "C" int passl_b200_grad_norm_finite(const float* g, long long n, float unscale, float clip_norm, float coef_max,
                                           int always_clip, float* ctrl, float* scratch, void* stream) {
  if (n <= 0 || n % 4 || !ctrl || !scratch) return PB_ERR_BAD_ARG;
  long long blocks = (n / 4 + 255) / 256;
  const int cap = num_sms() * 8;
  grad_norm_finite_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(g, n, unscale, clip_norm, coef_max,
                                                                                                always_clip, ctrl, scratch);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

static inline int opt_blocks(long long n) { return (int)((n + OPT_BLOCK - 1) / OPT_BLOCK); }

extern "C" int passl_b200_sgd_momentum(float* p, const float* g, float* v, void* p_bf16, float lr, float momentum, float wd,
                                       float grad_scale, const float* ctrl, long long n, void* stream) {
  if (n <= 0) return PB_OK;
  if (n % 4) return PB_ERR_BAD_ARG;
  sgd_momentum_kernel<<<opt_blocks(n), 256, 0, (cudaStream_t)stream>>>(p, g, v, reinterpret_cast<__nv_bfloat16*>(p_bf16), lr,
                                                                       momentum, wd, grad_scale, ctrl, n);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// norms: fp32 [2*num_segments] scratch (written here); block_seg: int32 [ceil(n/1024)]; seg_wd: fp32 [num_segments]
extern "C" int passl_b200_lars_momentum(float* p, const float* g, float* v, void* p_bf16, const int* block_seg,
                                        const float* seg_wd, float* norms, int num_segments, float lr, float momentum,
                                        float lars_coeff, float eps, float grad_scale, const float* ctrl, long long n,
                                        void* stream) {
  if (n <= 0) return PB_OK;
  if (n % OPT_BLOCK) return PB_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int nblocks = opt_blocks(n);
  float* part = nullptr;
  int rc = splitk_scratch(&part, (size_t)nblocks * 2, st);
  if (rc) return rc;
  seg_sqnorm_kernel<<<nblocks, 256, 0, st>>>(p, g, part, grad_scale, n);
  passl_b200_launch_counter_add(1);
  cudaError_t launched = cudaGetLastError();
  if (launched == cudaSuccess) {
    seg_norm_finalize_kernel<<<num_segments, 256, 0, st>>>(part, block_seg, nblocks, norms);
    passl_b200_launch_counter_add(1);
    launched = cudaGetLastError();
  }
  rc = splitk_release(part, st);
  if (launched != cudaSuccess) return (int)launched;
  if (rc) return rc;
  lars_momentum_kernel<<<opt_blocks(n), 256, 0, st>>>(p, g, v, reinterpret_cast<__nv_bfloat16*>(p_bf16), block_seg, norms, seg_wd,
                                                      lr, momentum, lars_coeff, eps, grad_scale, ctrl, n);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

extern "C" int passl_b200_adamw(float* p, const float* g, float* m, float* v, void* p_bf16, const int* block_seg,
                                const float* seg_wd, const float* seg_lr_ratio, float lr, float beta1, float beta2, float eps,
                                int step, float grad_scale, const float* ctrl, long long n, void* stream) {
  if (n <= 0) return PB_OK;
  if (n % 4 || step < 1) return PB_ERR_BAD_ARG;
  float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adamw_kernel<<<opt_blocks(n), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, reinterpret_cast<__nv_bfloat16*>(p_bf16), block_seg,
                                                                seg_wd, seg_lr_ratio, lr, beta1, beta2, eps, bc1, bc2,
                                                                grad_scale, ctrl, n);
  PB_LAUNCH_CHECK();
  return PB_OK;
}
