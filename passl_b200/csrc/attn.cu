// Fused multi-head self-attention for short sequences (ViT / MAE / CLIP towers: N <= 256 tokens, d = 64 or 32) on tcgen05.
//
//   S = Q K^T * d^-1/2  ->  softmax  ->  O = P V        per (batch, head); the [B,H,N,N] score tensor never reaches HBM
//   (the reference materialises it three times and keeps it for backward: passl/models/vision_transformer.py:145-153).
//
// Input is the packed output of the qkv Linear, qkv[b][n][s][h][e] (s = 0/1/2 for q/k/v) — exactly the reference's
// reshape [B,N,3,H,d] (vision_transformer.py:144-146) — read in place through a 4-D TMA tensor map (no permute pass).
// Output O[b][n][h][e] = [T, H*d] (the layout the proj Linear consumes) + LSE[b][h][n] (natural log) for the backward.
#include "common.cuh"
#include "host_utils.h"
#include "../../include/passl_b200.h"

#include <string.h>

namespace pb {

constexpr float kAttnLog2e = 1.4426950408889634f;
constexpr float kAttnLn2 = 0.6931471805599453f;

struct AttnParams {
  CUtensorMap qkv_map;   // dims (d, 3H, N, B), box {d, 1, 128, 1}
  CUtensorMap kv_map;    // same tensor, box {d, 1, NKP, 1}
  __nv_bfloat16* out;    // [B, N, H, d]
  float* lse;            // [B, H, N]
  int B, N, H, d;
  int NKP;               // keys padded to a multiple of 32 (<= 256)
  int mblocks;           // ceil(N / 128)
  int causal;
  float scale;
};

// ======================================================================================================================
// Forward, pipelined: load -> QK^T -> softmax -> PV -> epilogue strictly in sequence per (batch, head) ran at 114 TF/s at B=512,
// N=197, d=64.  One CTA (320 threads) keeps TWO work items (128 query rows of one head) in flight:
//   warp 0      : TMA producer — K / V of a head once (2-stage ring, shared by the head's query blocks), Q blocks (3-stage ring)
//   warp 1      : MMA issuer — S = Q K^T of item i, then O = P V of item i-1 (P read from TMEM as the A operand, V from shared
//                 memory as an MN-major B operand), so the tensor pipe works on one item while the SFUs work on the other
//   warps 2..5  : softmax group 0 (items 0, 2, 4, ...);  warps 6..9 : softmax group 1 (items 1, 3, 5, ...): one query row per
//                 thread, row max, exp2, P (bf16) written back over the S columns it was read from (tcgen05.st), then
//                 O / sum -> global.  Warps whose 32 rows are all beyond N only keep the barriers moving.
// TMEM: two 256-column slots; in a slot S uses [0, NKP), P (bf16x2) [0, NKP/2), O [128, 128 + d) — O is only written after P is
// complete, and the next S only after O has been read.
// Bound: N*NKP exponentials per head on 16 SFU lanes/clk/SM -> one 128-row item per 8*NKP cycles (1792 at NKP = 224), i.e. at
// most ~50 % of the tensor pipe; the QK^T + PV MMAs of an item take ~900 cycles.
// ======================================================================================================================
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__global__ void __launch_bounds__(320, 2) attn_fwd2_kernel(const __grid_constant__ AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int rowB = p.d * 2;                         // bytes per Q/K/V row (128 or 64)
  const uint32_t lt = (p.d == 64) ? 2u : 4u;        // SWIZZLE_128B / SWIZZLE_64B
  const uint32_t sbo = 8u * rowB;                   // 8-row atom stride
  constexpr int QST = 3, KVST = 2;
  const int kvB = ((p.NKP * rowB) + 1023) & ~1023;  // bytes of one K (or V) stage: NKP rows — short sequences leave room for 2 CTAs / SM
  const uint32_t slot_cols = (p.NKP <= 64) ? 128u : 256u, o_off = slot_cols / 2;   // TMEM: 2 slots; O sits in the upper half of a slot
  uint8_t* q_s = smem;                              // [QST][128][rowB]
  uint8_t* k_s = q_s + QST * 128 * rowB;            // [KVST][NKP][rowB]
  uint8_t* v_s = k_s + KVST * kvB;                  // [KVST][NKP][rowB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(v_s + KVST * kvB);
  uint64_t* q_full = bars;             // QST
  uint64_t* q_empty = q_full + QST;    // QST
  uint64_t* kv_full = q_empty + QST;   // KVST
  uint64_t* kv_empty = kv_full + KVST; // KVST
  uint64_t* s_full = kv_empty + KVST;  // 2
  uint64_t* p_full = s_full + 2;       // 2
  uint64_t* o_full = p_full + 2;       // 2
  uint64_t* slot_free = o_full + 2;    // 2
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(slot_free + 2);

  const uint32_t warp = warp_id(), lane = lane_id();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.qkv_map);
    tma_prefetch_desc(&p.kv_map);
    for (int i = 0; i < QST; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
    for (int i = 0; i < KVST; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&s_full[i], 1); mbar_init(&p_full[i], 4); mbar_init(&o_full[i], 1); mbar_init(&slot_free[i], 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 2 * slot_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int heads = p.B * p.H;

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    int qi = 0, kvi = 0;
    uint32_t qph = 0, kvph = 0;
    for (int head = blockIdx.x; head < heads; head += gridDim.x) {
      const int b = head / p.H, h = head - b * p.H;
      mbar_wait(&kv_empty[kvi], kvph ^ 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(&kv_full[kvi], (uint32_t)(2 * p.NKP * rowB));
        tma_load_4d(k_s + kvi * kvB, &p.kv_map, &kv_full[kvi], 0, p.H + h, 0, b);
        tma_load_4d(v_s + kvi * kvB, &p.kv_map, &kv_full[kvi], 0, 2 * p.H + h, 0, b);
      }
      __syncwarp();
      if (++kvi == KVST) { kvi = 0; kvph ^= 1; }
      for (int mb = 0; mb < p.mblocks; ++mb) {
        mbar_wait(&q_empty[qi], qph ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&q_full[qi], (uint32_t)(128 * rowB));
          tma_load_4d(q_s + qi * 128 * rowB, &p.qkv_map, &q_full[qi], 0, h, mb * 128, b);
        }
        __syncwarp();
        if (++qi == QST) { qi = 0; qph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    const uint32_t idesc1 = make_idesc_bf16(128, p.NKP, false, false);
    const uint32_t idesc2 = make_idesc_bf16(128, p.d, false, true);
    int qi = 0, kvi = 0, it = 0;
    uint32_t qph = 0, kvph = 0;
    int pv_slot = -1, pv_kv = 0, pv_last = 0;           // the item whose P V product is still to be issued
    uint32_t pv_ph = 0;
    auto issue_pv = [&]() {
      mbar_wait(&p_full[pv_slot], pv_ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t tm_p = tmem_base + pv_slot * slot_cols, tm_o = tm_p + o_off;
        const uint32_t va = smem_u32(v_s + pv_kv * kvB);
        for (int k = 0; k < p.NKP / 16; ++k)     // A: 16 keys = 8 packed columns of P; B: 16 key rows of V (MN-major, 2 atoms)
          umma_bf16_ts(tm_o, tm_p + k * 8, make_smem_desc(va + k * 16 * rowB, 0, sbo, lt), idesc2, k > 0 ? 1u : 0u);
        umma_commit(&o_full[pv_slot]);
        if (pv_last) umma_commit(&kv_empty[pv_kv]);
      }
      __syncwarp();
    };
    for (int head = blockIdx.x; head < heads; head += gridDim.x) {
      mbar_wait(&kv_full[kvi], kvph);
      for (int mb = 0; mb < p.mblocks; ++mb, ++it) {
        const int slot = it & 1;
        const uint32_t sph = (it >> 1) & 1;
        mbar_wait(&q_full[qi], qph);
        mbar_wait(&slot_free[slot], sph ^ 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t qa = smem_u32(q_s + qi * 128 * rowB), ka = smem_u32(k_s + kvi * kvB);
          for (int k = 0; k < p.d / 16; ++k)
            umma_bf16(tmem_base + slot * slot_cols, make_smem_desc(qa + k * 32, 16, sbo, lt), make_smem_desc(ka + k * 32, 16, sbo, lt), idesc1,
                      k > 0 ? 1u : 0u);
          umma_commit(&s_full[slot]);
          umma_commit(&q_empty[qi]);
        }
        __syncwarp();
        if (pv_slot >= 0) issue_pv();
        pv_slot = slot; pv_ph = sph; pv_kv = kvi; pv_last = (mb == p.mblocks - 1);
        if (++qi == QST) { qi = 0; qph ^= 1; }
      }
      if (++kvi == KVST) { kvi = 0; kvph ^= 1; }
    }
    if (pv_slot >= 0) issue_pv();
  } else {
    // ---------------- softmax / epilogue groups ----------------
    const int g = (warp - 2) >> 2;                    // group = TMEM slot
    const uint32_t q4 = warp & 3;                     // TMEM lane quarter of this warp
    const int r = q4 * 32 + lane;                     // row within the 128-row block
    const float c2 = p.scale * kAttnLog2e;
    const uint32_t ts = tmem_base + g * slot_cols + ((q4 * 32u) << 16);
    int it = 0;
    for (int head = blockIdx.x; head < heads; head += gridDim.x) {
      const int b = head / p.H, h = head - b * p.H;
      for (int mb = 0; mb < p.mblocks; ++mb, ++it) {
        if ((it & 1) != g) continue;
        const uint32_t sph = (it >> 1) & 1;
        const int row = mb * 128 + r;                 // query index
        const bool row_ok = row < p.N;
        const bool warp_ok = mb * 128 + (int)q4 * 32 < p.N;      // any valid row in this warp
        const int jmax = p.causal ? (row + 1 < p.N ? row + 1 : p.N) : p.N;   // valid keys: j < jmax
        mbar_wait(&s_full[g], sph);
        tc_fence_after();
        float l0 = 0.f, l1 = 0.f, m = 0.f;
        if (warp_ok) {
          // pass 1: row maximum of the raw scores (3-input max: 16 instructions per 32 columns)
          float m0 = -INFINITY, m1 = -INFINITY;
          for (int c = 0; c < p.NKP / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(ts + c * 32, v);
            tmem_ld_wait();
            if (c * 32 + 32 <= jmax) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                asm("max.f32 %0, %0, %1, %2;" : "+f"(m0) : "f"(__uint_as_float(v[j])), "f"(__uint_as_float(v[j + 1])));
                asm("max.f32 %0, %0, %1, %2;" : "+f"(m1) : "f"(__uint_as_float(v[j + 2])), "f"(__uint_as_float(v[j + 3])));
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (c * 32 + j < jmax) m0 = fmaxf(m0, __uint_as_float(v[j]));
            }
          }
          m = fmaxf(m0, m1);
          m = (!row_ok || m == -INFINITY) ? 0.f : m * c2;
          const float negm = -m;
          // pass 2: p = exp2(y - m), row sum, P (bf16x2) over the S columns already consumed.  O is normalised by the fp32 sum of
          // the unrounded probabilities (the bf16 rounding of P is unbiased: its effect on the sum is ~2^-9 / sqrt(N))
          for (int c = 0; c < p.NKP / 32; ++c) {
            uint32_t v[32], w[16];
            tmem_ld_32x32(ts + c * 32, v);
            tmem_ld_wait();
            if (c * 32 + 32 <= jmax) {
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                float p0, p1;
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p0) : "f"(fmaf(__uint_as_float(v[j]), c2, negm)));
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p1) : "f"(fmaf(__uint_as_float(v[j + 1]), c2, negm)));
                l0 += p0; l1 += p1;
                w[j >> 1] = pack_bf16x2(p0, p1);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                float p0 = (c * 32 + j < jmax) ? exp2f(fmaf(__uint_as_float(v[j]), c2, negm)) : 0.f;
                float p1 = (c * 32 + j + 1 < jmax) ? exp2f(fmaf(__uint_as_float(v[j + 1]), c2, negm)) : 0.f;
                l0 += p0; l1 += p1;
                w[j >> 1] = pack_bf16x2(p0, p1);
              }
            }
            tmem_st_32x16(ts + c * 16, w);
          }
          tmem_st_wait();
        }
        const float l = l0 + l1, l_exact = l;
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[g]);
        // epilogue: O / l
        mbar_wait(&o_full[g], sph);
        tc_fence_after();
        if (warp_ok) {
          const float inv = (l > 0.f) ? 1.f / l : 0.f;
          __nv_bfloat16* op = p.out + (((size_t)b * p.N + row) * p.H + h) * p.d;
          for (int c = 0; c < p.d / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(ts + o_off + c * 32, v);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
              for (int gq = 0; gq < 4; ++gq) {
                uint4 u;
                u.x = pack_bf16x2(__uint_as_float(v[gq * 8 + 0]) * inv, __uint_as_float(v[gq * 8 + 1]) * inv);
                u.y = pack_bf16x2(__uint_as_float(v[gq * 8 + 2]) * inv, __uint_as_float(v[gq * 8 + 3]) * inv);
                u.z = pack_bf16x2(__uint_as_float(v[gq * 8 + 4]) * inv, __uint_as_float(v[gq * 8 + 5]) * inv);
                u.w = pack_bf16x2(__uint_as_float(v[gq * 8 + 6]) * inv, __uint_as_float(v[gq * 8 + 7]) * inv);
                *reinterpret_cast<uint4*>(op + c * 32 + gq * 8) = u;
              }
            }
          }
          if (row_ok) p.lse[((size_t)b * p.H + h) * p.N + row] = (m + log2f(l_exact)) * kAttnLn2;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&slot_free[g]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, 2 * slot_cols);
  }
}

static int attn_make_maps(AttnParams& p, const void* qkv) {
  const uint64_t d = p.d, H3 = 3ull * p.H;
  uint64_t dims[4] = {d, H3, (uint64_t)p.N, (uint64_t)p.B};
  uint64_t str[3] = {d * 2, H3 * d * 2, (uint64_t)p.N * H3 * d * 2};
  uint32_t box_q[4] = {(uint32_t)p.d, 1, 128, 1};
  uint32_t box_kv[4] = {(uint32_t)p.d, 1, (uint32_t)p.NKP, 1};
  CUtensorMapSwizzle swz = (p.d == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  int rc = make_tmap_bf16(&p.qkv_map, qkv, 4, dims, str, box_q, swz);
  if (rc) return rc;
  return make_tmap_bf16(&p.kv_map, qkv, 4, dims, str, box_kv, swz);
}

}  // namespace pb

using namespace pb;

// qkv: bf16 [B, N, 3, H, d] (packed qkv Linear output);  out: bf16 [B, N, H, d];  lse: fp32 [B, H, N]
extern "C" int passl_b200_attention_fwd(const void* qkv, void* out, float* lse, int B, int N, int H, int d, float scale,
                                        int causal, void* stream) {
  if (B <= 0 || N <= 0 || N > 256 || H <= 0 || (d != 64 && d != 32)) return PB_ERR_UNSUPPORTED;
  if (reinterpret_cast<uintptr_t>(qkv) & 15) return PB_ERR_BAD_ARG;
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.out = reinterpret_cast<__nv_bfloat16*>(out); p.lse = lse;
  p.B = B; p.N = N; p.H = H; p.d = d; p.causal = causal; p.scale = scale;
  p.NKP = (N + 31) / 32 * 32;
  p.mblocks = (N + 127) / 128;
  int rc = attn_make_maps(p, qkv);
  if (rc) return rc;
  const int kvB = ((p.NKP * d * 2) + 1023) & ~1023;
  const int smem = 3 * 128 * d * 2 + 4 * kvB + 256 + 1024;
  static bool attr = false;
  if (!attr) {
    PB_CUDA_CHECK(cudaFuncSetAttribute(attn_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (3 * 128 + 4 * 256) * 128 + 256 + 1024));
    attr = true;
  }
  // short sequences: two CTAs per SM (shared memory and the 256-column TMEM allocation allow it) -> four items in flight per SM
  const int per_sm = (p.NKP <= 64 && smem <= 100 * 1024) ? 2 : 1;
  const int grid = B * H < num_sms() * per_sm ? B * H : num_sms() * per_sm;
  attn_fwd2_kernel<<<grid, 320, smem, (cudaStream_t)stream>>>(p);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// ======================================================================================================================
// Backward.  dqkv[b][n][s][h][e] (same packed layout as qkv) from dO[b][n][h][e], O, LSE.
//   S = Q K^T, P = exp(S*scale - lse), dP = dO V^T, dS = P o (dP - delta) * scale, delta_i = sum_e dO_ie O_ie
//   dV = P^T dO,  dK = dS^T Q,  dQ = dS K          (the reference keeps P in HBM; here it is recomputed per 128x128 tile)
// Tiles: query blocks i and key blocks j of 128.  TMEM: S [0,128) dP [128,256) dQ_0/dQ_1 [256,384) dK_j [384,448) dV_j [448,512).
// ======================================================================================================================
namespace pb {

struct AttnBwdParams {
  CUtensorMap qkv_map;   // dims (d, 3H, N, B), box {d, 1, 128, 1}
  CUtensorMap do_map;    // dims (d, H, N, B),  box {d, 1, 128, 1}
  const __nv_bfloat16* dO;
  const __nv_bfloat16* O;
  const float* lse;
  const float* delta;    // [B, H, N] fp32: sum_e dO * O per row, from attn_delta_kernel
  __nv_bfloat16* dqkv;
  int B, N, H, d, mblocks, causal;
  float scale;
};

// delta[b, h, n] = sum_e dO[b, n, h, e] * O[b, n, h, e].  One warp per token: the H*d contiguous elements of dO and O are read with
// coalesced 16-byte loads, each head's d elements sit in d / 8 neighbouring lanes (segmented shuffle reduction).  Round 2: inside
// the backward kernel this was a per-thread strided dot product at the start of every item — 15 % of the kernel's stall samples
// (`profiles/r02_ncu_attn_bwd_summary.txt`) with the DRAM latency fully exposed.
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ dO, const __nv_bfloat16* __restrict__ O,
                                                         float* __restrict__ delta, long long T, int N, int H, int d) {
  const long long tok = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (tok >= T) return;
  const int lane = threadIdx.x & 31;
  const int chunks = H * d / 8, seg = d / 8;
  const long long b = tok / N;
  const int n = (int)(tok - b * N);
  for (int c = lane; c < ((chunks + 31) / 32) * 32; c += 32) {
    float sacc = 0.f;
    if (c < chunks) {
      const uint4 ua = ld_nc_v4(dO + tok * (long long)H * d + c * 8), uo = ld_nc_v4(O + tok * (long long)H * d + c * 8);
      const float2 a0 = unpack_bf16x2(ua.x), a1 = unpack_bf16x2(ua.y), a2 = unpack_bf16x2(ua.z), a3 = unpack_bf16x2(ua.w);
      const float2 o0 = unpack_bf16x2(uo.x), o1 = unpack_bf16x2(uo.y), o2 = unpack_bf16x2(uo.z), o3 = unpack_bf16x2(uo.w);
      sacc = a0.x * o0.x + a0.y * o0.y + a1.x * o1.x + a1.y * o1.y + a2.x * o2.x + a2.y * o2.y + a3.x * o3.x + a3.y * o3.y;
    }
    for (int off = seg >> 1; off > 0; off >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, off);
    if (c < chunks && (c % seg) == 0) delta[(b * H + c / seg) * N + n] = sacc;
  }
}

// Round 2: EIGHT math warps (two per TMEM lane quarter, each takes two of the four 32-column chunks of a tile and half of the
// dK / dV / dQ epilogue columns) + the control warp: the softmax arithmetic between the two MMA groups of a tile was half of the
// tile time with one warp per sub-partition.
constexpr int kAttnBwdThreads = 288;
__global__ void __launch_bounds__(kAttnBwdThreads, 1) attn_bwd_kernel(const __grid_constant__ AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int rowB = p.d * 2;
  const uint32_t lt = (p.d == 64) ? 2u : 4u;
  const uint32_t sbo = 8u * rowB;
  uint8_t* q_s = smem;
  uint8_t* k_s = q_s + 256 * rowB;
  uint8_t* v_s = k_s + 256 * rowB;
  uint8_t* do_s = v_s + 256 * rowB;
  uint8_t* p_s = do_s + 256 * rowB;          // 2 chunks x [128][128 B]
  uint8_t* ds_s = p_s + 2 * 128 * 128;       // 2 chunks x [128][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(ds_s + 2 * 128 * 128);
  uint64_t* load_full = bars;       // tx
  uint64_t* sp_full = bars + 1;     // S and dP ready            (MMA commit)
  uint64_t* pd_full = bars + 2;     // P and dS written to smem   (4 warp arrivals)
  uint64_t* kv_done = bars + 3;     // dK_j, dV_j complete        (MMA commit)
  uint64_t* kv_free = bars + 4;     // dK_j, dV_j read out        (4 warp arrivals)
  uint64_t* q_done = bars + 5;      // dQ complete                (MMA commit)
  uint64_t* q_free = bars + 6;      // dQ read out                (4 warp arrivals)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 7);

  const uint32_t warp = warp_id(), lane = lane_id();
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&p.qkv_map);
    tma_prefetch_desc(&p.do_map);
    mbar_init(load_full, 1);
    mbar_init(sp_full, 1);
    mbar_init(pd_full, 8);
    mbar_init(kv_done, 1);
    mbar_init(kv_free, 8);
    mbar_init(q_done, 1);
    mbar_init(q_free, 8);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const uint32_t tm_s = tmem_base, tm_dp = tmem_base + 128, tm_dq = tmem_base + 256, tm_dk = tmem_base + 384,
                 tm_dv = tmem_base + 448;
  const int items = p.B * p.H;
  const int nb = p.mblocks;
  uint32_t ph_load = 0, ph_sp = 0, ph_pd = 0, ph_kvd = 0, ph_kvf = 0, ph_qd = 0, ph_qf = 0;

  if (warp == 8) {
    {   // warp-uniform control loop; TMA / tcgen05 issue elect-predicated
      // Tiles are cut to the valid extent of the sequence (N = 197: the second block has 69 rows / keys, N = 50: one 64-key
      // tile): S / dP over the valid keys rounded up to 32, dV / dK over the valid query rows rounded up to 16, dQ over the
      // valid keys — the padded remainder is neither multiplied nor exponentiated.
      const uint32_t id_kv = make_idesc_bf16(128, p.d, true, true);
      const uint32_t id_q = make_idesc_bf16(128, p.d, false, true);
      bool first_item = true;
      for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int b = item / p.H, h = item - b * p.H;
        // previous item's MMAs are all complete (q_done waited below), epilogue reads are TMEM-only -> smem reusable
        if (elect_one()) {
          mbar_arrive_expect_tx(load_full, (uint32_t)(4 * nb * 128 * rowB));
          for (int mb = 0; mb < nb; ++mb) {
            tma_load_4d(q_s + mb * 128 * rowB, &p.qkv_map, load_full, 0, h, mb * 128, b);
            tma_load_4d(k_s + mb * 128 * rowB, &p.qkv_map, load_full, 0, p.H + h, mb * 128, b);
            tma_load_4d(v_s + mb * 128 * rowB, &p.qkv_map, load_full, 0, 2 * p.H + h, mb * 128, b);
            tma_load_4d(do_s + mb * 128 * rowB, &p.do_map, load_full, 0, h, mb * 128, b);
          }
        }
        __syncwarp();
        mbar_wait(load_full, ph_load); ph_load ^= 1;
        tc_fence_after();
        if (!first_item) { mbar_wait(q_free, ph_qf); ph_qf ^= 1; }   // dQ accumulators of the previous item were read out
        for (int j = 0; j < nb; ++j) {
          if (!(first_item && j == 0)) { mbar_wait(kv_free, ph_kvf); ph_kvf ^= 1; }   // dK/dV accumulators read out
          for (int i = 0; i < nb; ++i) {
            const uint32_t qa = smem_u32(q_s + i * 128 * rowB), doa = smem_u32(do_s + i * 128 * rowB);
            const uint32_t ka = smem_u32(k_s + j * 128 * rowB), va = smem_u32(v_s + j * 128 * rowB);
            const int nk = p.N - j * 128 < 128 ? p.N - j * 128 : 128, nr = p.N - i * 128 < 128 ? p.N - i * 128 : 128;
            const int nmma = ((nk + 31) / 32) * 32, rk = (nr + 15) / 16;
            const uint32_t id_s = make_idesc_bf16(128, (uint32_t)nmma, false, false);
            if (elect_one()) {
              for (int k = 0; k < p.d / 16; ++k)
                umma_bf16(tm_s, make_smem_desc(qa + k * 32, 16, sbo, lt), make_smem_desc(ka + k * 32, 16, sbo, lt), id_s, k > 0);
              for (int k = 0; k < p.d / 16; ++k)
                umma_bf16(tm_dp, make_smem_desc(doa + k * 32, 16, sbo, lt), make_smem_desc(va + k * 32, 16, sbo, lt), id_s, k > 0);
              umma_commit(sp_full);
            }
            __syncwarp();
            mbar_wait(pd_full, ph_pd); ph_pd ^= 1;
            tc_fence_after();
            const uint32_t pa = smem_u32(p_s), dsa = smem_u32(ds_s);
            if (elect_one()) {
            for (int k = 0; k < rk; ++k) {   // K = the valid query rows
              // dV_j += P^T dO_i ; dK_j += dS^T Q_i      (A = P / dS viewed MN-major: M = keys, K = query rows)
              umma_bf16(tm_dv, make_smem_desc(pa + k * 2048, 128 * 128, 1024, 2), make_smem_desc(doa + k * 16 * rowB, 0, sbo, lt),
                        id_kv, (i > 0 || k > 0));
              umma_bf16(tm_dk, make_smem_desc(dsa + k * 2048, 128 * 128, 1024, 2), make_smem_desc(qa + k * 16 * rowB, 0, sbo, lt),
                        id_kv, (i > 0 || k > 0));
            }
            for (int k = 0; k < nmma / 16; ++k)     // dQ_i += dS K_j   (A = dS K-major over the valid keys, B = K_j MN-major)
              umma_bf16(tm_dq + i * 64, make_smem_desc_sw128(dsa + (k >> 2) * (128 * 128) + (k & 3) * 32, 16, 1024),
                        make_smem_desc(ka + k * 16 * rowB, 0, sbo, lt), id_q, (j > 0 || k > 0));
            if (i == nb - 1) umma_commit(kv_done);
            if (i == nb - 1 && j == nb - 1) umma_commit(q_done);
            }
            __syncwarp();
          }
        }
        // all MMAs of this item retired before the next item's TMA overwrites shared memory
        // (q_done is also consumed by the epilogue warps; this thread waits one phase behind at most)
        mbar_wait(q_done, ph_qd); ph_qd ^= 1;
        first_item = false;
      }
    }
  } else {
    const uint32_t q4 = warp & 3u, hf = warp >> 2;     // TMEM lane quarter, column half
    const int r = q4 * 32 + lane;
    const float c2 = p.scale * kAttnLog2e;
    const uint32_t lane_off = (q4 * 32u) << 16;
    float nlse[2] = {0.f, 0.f}, ndel[2] = {0.f, 0.f};
    auto load_consts = [&](int item_) {
      if (item_ >= items) return;
      for (int i = 0; i < nb; ++i) {
        const int row = i * 128 + r;
        nlse[i] = 0.f; ndel[i] = 0.f;
        if (row < p.N) {
          nlse[i] = p.lse[(size_t)item_ * p.N + row];
          ndel[i] = p.delta[(size_t)item_ * p.N + row];
        }
      }
    };
    load_consts((int)blockIdx.x);
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int b = item / p.H, h = item - b * p.H;
      // per-row constants for both query blocks: lse (log2 domain) and delta — requested one item ahead
      float lse2[2], delta[2];
      for (int i = 0; i < 2; ++i) { lse2[i] = nlse[i] * kAttnLog2e; delta[i] = ndel[i]; }
      load_consts(item + (int)gridDim.x);
      for (int j = 0; j < nb; ++j) {
        for (int i = 0; i < nb; ++i) {
          const int row = i * 128 + r;
          const bool row_ok = row < p.N;
          const int nk = p.N - j * 128 < 128 ? p.N - j * 128 : 128, nr = p.N - i * 128 < 128 ? p.N - i * 128 : 128;
          const int kc = (nk + 31) / 32;                                   // 32-key chunks the MMAs produced
          const bool warp_live = (int)q4 * 32 < ((nr + 15) / 16) * 16;     // rows the dV / dK MMAs will read
          mbar_wait(sp_full, ph_sp); ph_sp ^= 1;
          tc_fence_after();
          for (int c = (int)hf; c < kc && warp_live; c += 2) {
            uint32_t sv[32], dv[32];
            tmem_ld_32x32(tm_s + lane_off + c * 32, sv);
            tmem_ld_32x32(tm_dp + lane_off + c * 32, dv);
            tmem_ld_wait();
            float pe[32], de[32];
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) {
              const int key = j * 128 + c * 32 + jj;
              const bool ok = row_ok && key < p.N && (!p.causal || key <= row);
              const float pv = ok ? exp2f(__uint_as_float(sv[jj]) * c2 - lse2[i]) : 0.f;
              pe[jj] = pv;
              de[jj] = pv * (__uint_as_float(dv[jj]) - delta[i]) * p.scale;
            }
            const int chunk = c >> 1;
            const uint32_t roff = chunk * (128 * 128) + (r >> 3) * 1024 + (r & 7) * 128;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const int j8 = ((c * 32) & 63) + g * 8;
              const uint32_t off = roff + ((((j8 >> 3) ^ (r & 7)) & 7) << 4);
              uint4 u, w;
              u.x = pack_bf16x2(pe[g * 8 + 0], pe[g * 8 + 1]); u.y = pack_bf16x2(pe[g * 8 + 2], pe[g * 8 + 3]);
              u.z = pack_bf16x2(pe[g * 8 + 4], pe[g * 8 + 5]); u.w = pack_bf16x2(pe[g * 8 + 6], pe[g * 8 + 7]);
              w.x = pack_bf16x2(de[g * 8 + 0], de[g * 8 + 1]); w.y = pack_bf16x2(de[g * 8 + 2], de[g * 8 + 3]);
              w.z = pack_bf16x2(de[g * 8 + 4], de[g * 8 + 5]); w.w = pack_bf16x2(de[g * 8 + 6], de[g * 8 + 7]);
              *reinterpret_cast<uint4*>(p_s + off) = u;
              *reinterpret_cast<uint4*>(ds_s + off) = w;
            }
          }
          tc_fence_before();
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(pd_full);
        }
        // dK_j / dV_j epilogue: TMEM lane = key row
        mbar_wait(kv_done, ph_kvd); ph_kvd ^= 1;
        tc_fence_after();
        {
          const int key = j * 128 + r;
          __nv_bfloat16* dk = p.dqkv + ((((size_t)b * p.N + key) * 3 + 1) * p.H + h) * p.d;
          __nv_bfloat16* dvp = p.dqkv + ((((size_t)b * p.N + key) * 3 + 2) * p.H + h) * p.d;
          for (int c = (int)hf; c < p.d / 32; c += 2) {
            uint32_t a[32], bq[32];
            tmem_ld_32x32(tm_dk + lane_off + c * 32, a);
            tmem_ld_32x32(tm_dv + lane_off + c * 32, bq);
            tmem_ld_wait();
            if (key < p.N) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                uint4 u, w;
                u.x = pack_bf16x2(__uint_as_float(a[g * 8 + 0]), __uint_as_float(a[g * 8 + 1]));
                u.y = pack_bf16x2(__uint_as_float(a[g * 8 + 2]), __uint_as_float(a[g * 8 + 3]));
                u.z = pack_bf16x2(__uint_as_float(a[g * 8 + 4]), __uint_as_float(a[g * 8 + 5]));
                u.w = pack_bf16x2(__uint_as_float(a[g * 8 + 6]), __uint_as_float(a[g * 8 + 7]));
                w.x = pack_bf16x2(__uint_as_float(bq[g * 8 + 0]), __uint_as_float(bq[g * 8 + 1]));
                w.y = pack_bf16x2(__uint_as_float(bq[g * 8 + 2]), __uint_as_float(bq[g * 8 + 3]));
                w.z = pack_bf16x2(__uint_as_float(bq[g * 8 + 4]), __uint_as_float(bq[g * 8 + 5]));
                w.w = pack_bf16x2(__uint_as_float(bq[g * 8 + 6]), __uint_as_float(bq[g * 8 + 7]));
                *reinterpret_cast<uint4*>(dk + c * 32 + g * 8) = u;
                *reinterpret_cast<uint4*>(dvp + c * 32 + g * 8) = w;
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(kv_free);
      }
      // dQ epilogue
      mbar_wait(q_done, ph_qd); ph_qd ^= 1;
      tc_fence_after();
      for (int i = 0; i < nb; ++i) {
        const int row = i * 128 + r;
        __nv_bfloat16* dq = p.dqkv + ((((size_t)b * p.N + row) * 3 + 0) * p.H + h) * p.d;
        for (int c = (int)hf; c < p.d / 32; c += 2) {
          uint32_t a[32];
          tmem_ld_32x32(tm_dq + i * 64 + lane_off + c * 32, a);
          tmem_ld_wait();
          if (row < p.N) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              uint4 u;
              u.x = pack_bf16x2(__uint_as_float(a[g * 8 + 0]), __uint_as_float(a[g * 8 + 1]));
              u.y = pack_bf16x2(__uint_as_float(a[g * 8 + 2]), __uint_as_float(a[g * 8 + 3]));
              u.z = pack_bf16x2(__uint_as_float(a[g * 8 + 4]), __uint_as_float(a[g * 8 + 5]));
              u.w = pack_bf16x2(__uint_as_float(a[g * 8 + 6]), __uint_as_float(a[g * 8 + 7]));
              *reinterpret_cast<uint4*>(dq + c * 32 + g * 8) = u;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(q_free);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace pb

// dO, O: bf16 [B, N, H, d]; lse fp32 [B, H, N]; dqkv: bf16 [B, N, 3, H, d] (fully overwritten)
// delta_ws: fp32 [B, H, N] workspace (row sums of dO * O, written by a pre-pass on the same stream)
extern "C" int passl_b200_attention_bwd(const void* qkv, const void* dO, const void* O, const float* lse, void* dqkv, float* delta_ws,
                                        int B, int N, int H, int d, float scale, int causal, void* stream) {
  if (B <= 0 || N <= 0 || N > 256 || H <= 0 || (d != 64 && d != 32) || !delta_ws) return PB_ERR_UNSUPPORTED;
  AttnBwdParams p;
  memset(&p, 0, sizeof(p));
  p.dO = reinterpret_cast<const __nv_bfloat16*>(dO); p.O = reinterpret_cast<const __nv_bfloat16*>(O);
  p.lse = lse; p.dqkv = reinterpret_cast<__nv_bfloat16*>(dqkv);
  p.delta = delta_ws;
  p.B = B; p.N = N; p.H = H; p.d = d; p.causal = causal; p.scale = scale;
  p.mblocks = (N + 127) / 128;
  CUtensorMapSwizzle swz = (d == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  {
    const uint64_t dd = d, H3 = 3ull * H;
    uint64_t dims[4] = {dd, H3, (uint64_t)N, (uint64_t)B};
    uint64_t str[3] = {dd * 2, H3 * dd * 2, (uint64_t)N * H3 * dd * 2};
    uint32_t box[4] = {(uint32_t)d, 1, 128, 1};
    int rc = make_tmap_bf16(&p.qkv_map, qkv, 4, dims, str, box, swz);
    if (rc) return rc;
    uint64_t dims2[4] = {dd, (uint64_t)H, (uint64_t)N, (uint64_t)B};
    uint64_t str2[3] = {dd * 2, (uint64_t)H * dd * 2, (uint64_t)N * H * dd * 2};
    rc = make_tmap_bf16(&p.do_map, dO, 4, dims2, str2, box, swz);
    if (rc) return rc;
  }
  const int smem = 4 * 256 * d * 2 + 4 * 128 * 128 + 256 + 1024;
  static bool attr = false;
  if (!attr) {
    PB_CUDA_CHECK(cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * 256 * 128 + 4 * 128 * 128 + 256 + 1024));
    attr = true;
  }
  const long long T = (long long)B * N;
  attn_delta_kernel<<<(unsigned)((T + 7) / 8), 256, 0, (cudaStream_t)stream>>>(p.dO, p.O, delta_ws, T, N, H, d);
  PB_LAUNCH_CHECK();
  int grid = B * H < num_sms() ? B * H : num_sms();
  attn_bwd_kernel<<<grid, kAttnBwdThreads, smem, (cudaStream_t)stream>>>(p);
  PB_LAUNCH_CHECK();
  return PB_OK;
}
