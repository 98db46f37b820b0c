// passl_b200 — persistent warp-specialised tcgen05 GEMM / implicit-GEMM kernel for sm_100a.
//
//   D[m, n] = epilogue( alpha * sum_k A[m, k] * B[n, k] )         bf16 inputs, fp32 accumulation in TMEM
//
// One kernel serves every dense contraction on the PASSL hot path (SURVEY.md §8 a1/a3/a4, App. A):
//   * Linear fwd / dgrad / wgrad (ViT qkv/proj/fc1/fc2, necks, patch-embed, 1x1 convs)      -> MAT operands
//   * 3x3 / strided convolution fwd + dgrad as implicit GEMM over NHWC activations             -> PATCH_K  A operand
//   * convolution wgrad (K = output pixels, both operands channel-contiguous)                  -> PATCH_MN operands
//
// Structure (one persistent CTA per SM, 320 threads):
//   warp 0      : TMA producer  — cp.async.bulk.tensor into a STAGES-deep smem ring (SWIZZLE_128B); warp-uniform loop, the
//                                 issue itself predicated on elect.sync
//   warp 1      : MMA issuer    — tcgen05.mma cta_group::1, M=128, N=BN, K=16 per instruction (elect.sync-predicated)
//   warps 2..9  : epilogue      — two warps per TMEM lane quarter split the 32-column chunks: tcgen05.ld TMEM->regs,
//                                 bias / activation / gate, bf16 tile staged through padded smem for row-coalesced residual
//                                 loads and stores, optional BatchNorm statistics of the stored values, fp32 / atomic path
// TMEM holds two BN-column accumulators so the epilogue of tile i overlaps the main loop of tile i+1.
#pragma once
#include "common.cuh"

namespace pb {

enum OperandMode : int {
  OP_MAT_K = 0,     // 2D matrix [rows, K], K contiguous            (tensor map dims: K, rows)
  OP_MAT_MN = 1,    // 2D matrix [K, rows], rows contiguous         (tensor map dims: rows, K)
  OP_PATCH_K = 2,   // NHWC activation patch, channels = K slice    (tensor map dims: C, W, H, N)
  OP_PATCH_MN = 3,  // NHWC activation patch, pixels = K, channels = rows
};
enum ActMode : int { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2, ACT_QUICKGELU = 3 };

constexpr int kMaxTaps = 12;
constexpr int kEpiWarps = 8;                       // epilogue warps (2 per TMEM lane quarter)
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;  // warp 0 TMA, warp 1 MMA, warps 2.. epilogue
// HALO variant (3x3 stride-1 convolutions): pixel tile 16 rows x 8 columns; ONE TMA box {64 ch, 10, 18} per 64-channel chunk holds
// every pixel the nine taps touch; tap (r, s) is the K-major view that starts (r * 10 + s) pixel rows into the box, 8-pixel row
// groups 10 pixels (1280 B) apart (descriptor semantics pinned by umma_probe.cu: shifted start, SBO = 1280, base_offset 0).
constexpr int kHaloTH = 16, kHaloTW = 8, kHaloW = kHaloTW + 2, kHaloRows = (kHaloTH + 2) * kHaloW;   // 180 pixel rows of 128 B
constexpr int kHaloBytes = 23 * 1024;              // 180 * 128 = 23040 rounded up to a 1024 multiple
constexpr int kHaloStages = 2;
constexpr int kEpiStride = 80;                     // bytes per staged row: 32 bf16 + 16 B pad (conflict-free 16 B accesses)


struct PatchGeom {
  int TN, TH, TW;    // patch box: images x rows x cols  (TN*TH*TW <= 128)
  int nb, hb, wb;    // number of patches along each axis
  int Nimg, Ho, Wo;  // bounds of the pixel grid the patches enumerate
};

struct GemmOperand {
  CUtensorMap maps[4];  // [0] always valid; [1..3] parity maps for stride-2 sources
  int mode;
  int cchunks;          // PATCH_K: 64-channel chunks per tap
  int tx_bytes;         // bytes one stage load of this operand deposits
  int ntaps;
  signed char dh[kMaxTaps], dw[kMaxTaps], map[kMaxTaps];  // per-tap coordinate shift + parity map
};

struct GemmParams {
  GemmOperand a, b;
  PatchGeom geom;       // used when an operand is PATCH_* or out_pixel != 0
  int M, N;             // logical output extent (rows, cols)
  int m_blocks, n_blocks, splits;
  int k_iters;          // total pipeline iterations over K (all taps / chunks / pixel patches)
  int k_steps;          // UMMA (K=16) steps per pipeline iteration
  // N-tile decode for wgrad: n_blk -> (tap, channel block)
  int n_blocks_per_tap; // 0 => plain
  int n_per_tap;        // Cin (columns per tap) when n_blocks_per_tap > 0
  // epilogue
  void* out;
  long long ldc;        // elements between consecutive output rows (pixels)
  int out_fp32;         // 0: bf16, 1: fp32
  int atomic_add;       // fp32 only: red.add instead of store (split-K / wgrad)
  float* partial;       // atomic_add with splits > 1: split s stores its tile to partial + s * part_stride (same
  long long part_stride; // addressing as out); splitk_reduce adds the slices into out in split order
  int out_pixel;        // 1: row -> NHWC pixel address through geom + (OH, OW, osh, osw, oh0, ow0)
  int OH, OW, osh, osw, oh0, ow0;
  const float* bias;            // [N] or null
  const __nv_bfloat16* residual;  // same addressing as out (bf16) or null
  int act;
  float alpha;
  // optional gate applied after the activation: 1 = ReLU mask (aux > 0), 2 = multiply by GELU'(aux), 3 = QuickGELU'(aux)
  const __nv_bfloat16* aux;     // same addressing as out
  int aux_mode;
  __nv_bfloat16* preact;        // optional: value before the activation (bias added), same addressing as out (GELU backward)
  // optional per-column statistics of the stored bf16 value (BatchNorm batch stats): partials [4 * gridDim.x][2][N] (sum, sum of
  // squares), zero-initialised by the host; row 4*b + q is only touched by the two epilogue warps of lane quarter q of CTA b, on
  // disjoint columns -> no atomics, deterministic per grid
  float* col_sum;
  // residual through the tensor pipe: when res_iters > 0 the producer appends res_iters (= 128 / 64) pipeline iterations per tile
  // that load an identity slice as A and the residual tile (MN-major) as B, so that D += I * R — the residual is prefetched as
  // deep as the operands (a register prefetch in the epilogue cannot cover the ~4 us DRAM latency of a saturated HBM)
  CUtensorMap res_map, eye_map;
  int res_iters;
  // EPI = 1 (plain row-major bf16 outputs of the linear layers): 32 x 32 output boxes leave through TMA stores
  CUtensorMap out_map, pre_map;
  // the epilogue's operand tile (gate operand / residual) of a whole output tile, requested into L2 by the producer one tile
  // ahead of the epilogue (box BN x 128): the epilogue's own one-chunk-ahead register prefetch then only sees L2 latency
  CUtensorMap tile_map;
  int tile_prefetch;
  int halo_dh0, halo_dw0;   // HALO variant: smallest row / column shift over the taps = origin of the halo box relative to the tile
};

// EW = number of epilogue warps: 8 (two per TMEM lane quarter), or 16 for the epilogue-bound linear launches (GELU / gate
// arithmetic): four warps per sub-partition hide the MUFU / TMEM / shared-memory latencies that two cannot; 576 threads leave 112
// registers per thread, so that variant reads the accumulator in place (no read-ahead) and pays for its 64 KB of staging tiles
// with one pipeline stage.
template <int BN, int BK, bool A_MN, bool B_MN, int EPI = 0, int CG = 1, bool HALO = false, int EW = kEpiWarps>
struct GemmSmem {
  static constexpr int BM = 128;
  static constexpr int A_BYTES = HALO ? 0 : BM * BK * 2;     // HALO: the A operand lives in its own ring of halo boxes (after the stages)
  static constexpr int AH_BYTES = HALO ? kHaloStages * kHaloBytes : 0;
  static constexpr int B_BYTES = BN * BK * 2 / CG;   // CTA pair (CG = 2): each CTA holds BN / 2 rows of the B tile
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BUDGET = 196 * 1024 - AH_BYTES - (EW > 8 ? (EW - 8) * 4096 : 0);
  static constexpr int STAGES_RAW = BUDGET / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int BAR_BYTES = 256;
  static constexpr int BIAS_BYTES = EW * 4 * 32 * 4;              // per-warp bias slices of the current tile (4 chunks x 32 columns, fp32)
  // EPI 0: per-warp padded staging tiles + bias slices, after the barriers.  EPI 1, 2: per warp two dense 2 KB tiles (32 rows x
  // 64 B, SWIZZLE_64B, the source of the TMA stores) placed right after the stages so that they stay 1024-byte aligned.
  static constexpr int EPI_BYTES = EPI >= 1 ? EW * 4096 : EW * 32 * kEpiStride + BIAS_BYTES;
  static constexpr int AH_OFF = STAGES * STAGE_BYTES;
  static constexpr int EPI_OFF = EPI >= 1 ? AH_OFF + AH_BYTES : AH_OFF + AH_BYTES + BAR_BYTES;
  static constexpr int BAR_OFF = EPI >= 1 ? AH_OFF + AH_BYTES + EPI_BYTES : AH_OFF + AH_BYTES;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + AH_BYTES + BAR_BYTES + EPI_BYTES + 1024;  // + alignment slack
  static constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static_assert(TOTAL <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void decode_patch(const PatchGeom& g, int idx, int& n0, int& h0, int& w0) {
  int iw = idx % g.wb;
  int t = idx / g.wb;
  int ih = t % g.hb;
  int in_ = t / g.hb;
  n0 = in_ * g.TN;
  h0 = ih * g.TH;
  w0 = iw * g.TW;
}

// Phi(x) = 0.5 * erfc(-x / sqrt 2) for the exact (erf) GELU of the reference, and e = exp(-x^2 / 2) for its derivative.
// erfc(z) = t * (a1 + t * (a2 + ... a5 t)) * exp(-z^2), t = 1 / (1 + 0.3275911 z), z >= 0 (Abramowitz & Stegun 7.1.26, absolute
// error < 1.5e-7, the tail is formed without cancellation): 2 MUFU (rcp, ex2) + 10 FMA-pipe instructions.  erff() costs ~3x that
// and, inlined 32x per chunk, pushed the epilogue out of the instruction cache (fc1 of ViT-B ran at 300 TF/s, profiles/
// r02_vit_gemm_probe.txt).
// Eight elements at a time, stage by stage, so that the eight MUFU.RCP / MUFU.EX2 are in flight together (written one element
// at a time ptxas chained rcp -> Horner -> ex2 through one register and every element paid the MUFU latency: short-scoreboard
// stalls were half of the epilogue of fc1, profiles/r02_ncu_vitgemm_summary.txt).
__device__ __forceinline__ void gelu_phi8(const float* x, float* ph, float* e) {
  float t[8], y[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(t[k]) : "f"(fmaf(0.3275911f * 0.70710678118654752f, fabsf(x[k]), 1.f)));
#pragma unroll
  for (int k = 0; k < 8; ++k) asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(e[k]) : "f"(x[k] * x[k] * -0.72134752044448170f));
#pragma unroll
  for (int k = 0; k < 8; ++k) y[k] = fmaf(1.061405429f, t[k], -1.453152027f);
#pragma unroll
  for (int k = 0; k < 8; ++k) y[k] = fmaf(y[k], t[k], 1.421413741f);
#pragma unroll
  for (int k = 0; k < 8; ++k) y[k] = fmaf(y[k], t[k], -0.284496736f);
#pragma unroll
  for (int k = 0; k < 8; ++k) y[k] = fmaf(y[k], t[k], 0.254829592f);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float h = 0.5f * (y[k] * t[k]) * e[k];   // Phi(-|x|)
    ph[k] = x[k] < 0.f ? h : 1.f - h;
  }
}
__device__ __forceinline__ void act_gelu8(float* f) {
  float ph[8], e[8];
  gelu_phi8(f, ph, e);
#pragma unroll
  for (int k = 0; k < 8; ++k) f[k] *= ph[k];
}
__device__ __forceinline__ float act_quickgelu(float v) { return v / (1.f + __expf(-1.702f * v)); }
// f *= d/da gelu(a) at the saved pre-activation a.  With u = |a| sqrt(log2(e) / 2), e = 2^(-u^2) = exp(-a^2 / 2) and the 3-term
// A&S 7.1.25 form of erfc (|error| < 2.5e-5; the gate is exact to 1.1e-5, checked against erf on [-8, 8]):
//   s = gelu'(-|a|) = Phi(-|a|) - |a| phi(a) = e * (t (a1 + t (a2 + a3 t)) / 2 - u / sqrt(pi log2 e)),   t = 1 / (1 + p u)
//   gelu'(a) = a < 0 ? s : 1 - s            (gelu'(a) + gelu'(-a) = 1)
// 11 FMA-pipe instructions + 2 MUFU per element; the epilogue of fc2's dgrad is issue-bound on this arithmetic.
__device__ __forceinline__ void gate_gelu8(float* f, const float* a) {
  float t[8], e[8], u[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) u[k] = fabsf(a[k]) * 0.8493218002880191f;
#pragma unroll
  for (int k = 0; k < 8; ++k) asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(t[k]) : "f"(fmaf(0.39169196791136207f, u[k], 1.f)));
#pragma unroll
  for (int k = 0; k < 8; ++k) asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(e[k]) : "f"(-(u[k] * u[k])));
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    float y = fmaf(0.5f * 0.7478556f, t[k], 0.5f * -0.0958798f);
    y = fmaf(y, t[k], 0.5f * 0.3480242f);
    const float w = fmaf(-0.46971863934982566f, u[k], y * t[k]);
    const float fs = f[k] * (w * e[k]);
    f[k] = a[k] < 0.f ? fs : f[k] - fs;
  }
}
__device__ __forceinline__ float gate_quickgelu(float a) {
  const float sg = 1.f / (1.f + __expf(-1.702f * a));
  return sg * (1.f + 1.702f * a * (1.f - sg));
}
// the gate of one 8-column group of a row (aux values packed as bf16), mode fixed per call so that only the taken variant is
// in the instruction stream that is executed
template <int MODE>
__device__ __forceinline__ void apply_gate8(float* f, const uint4& u) {
  const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
  const float a[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
  if (MODE == 2) {
    gate_gelu8(f, a);
    return;
  }
  if (MODE == 4) {      // plain residual add
#pragma unroll
    for (int ee = 0; ee < 8; ++ee) f[ee] += a[ee];
    return;
  }
#pragma unroll
  for (int ee = 0; ee < 8; ++ee) {
    if (MODE == 1) f[ee] = a[ee] > 0.f ? f[ee] : 0.f;
    else f[ee] *= gate_quickgelu(a[ee]);
  }
}

// Issue the TMA loads of one pipeline stage for one operand.
//   row_blk : index of the 128-row (A) / BN-row (B) block, or patch index in PATCH_K mode
//   kit     : pipeline iteration
template <int CG>
__device__ __forceinline__ void tma2(void* d, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  if constexpr (CG == 2) tma_load_2d_pair(d, m, bar, c0, c1);
  else tma_load_2d(d, m, bar, c0, c1);
}
template <int CG>
__device__ __forceinline__ void tma4(void* d, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  if constexpr (CG == 2) tma_load_4d_pair(d, m, bar, c0, c1, c2, c3);
  else tma_load_4d(d, m, bar, c0, c1, c2, c3);
}

template <int ROWS, int BK, int CG = 1>
__device__ __forceinline__ void issue_operand_load(const GemmOperand& op, const PatchGeom& g, uint8_t* dst,
                                                   uint64_t* bar, int row0, int patch_idx, int tap_fixed,
                                                   int kit) {
  if (op.mode == OP_MAT_K) {
    tma2<CG>(dst, &op.maps[0], bar, kit * BK, row0);
  } else if (op.mode == OP_MAT_MN) {
#pragma unroll
    for (int j = 0; j < ROWS / 64; ++j) tma2<CG>(dst + j * (BK * 128), &op.maps[0], bar, row0 + 64 * j, kit * BK);
  } else if (op.mode == OP_PATCH_K) {
    int tap = kit / op.cchunks;
    int cc = kit - tap * op.cchunks;
    int n0, h0, w0;
    decode_patch(g, patch_idx, n0, h0, w0);
    tma4<CG>(dst, &op.maps[op.map[tap]], bar, cc * 64, w0 + op.dw[tap], h0 + op.dh[tap], n0);
  } else {  // OP_PATCH_MN: K = pixels of patch `kit`, rows = channels starting at row0
    int n0, h0, w0;
    decode_patch(g, kit, n0, h0, w0);
    int tap = tap_fixed;
#pragma unroll
    for (int j = 0; j < ROWS / 64; ++j)
      tma4<CG>(dst + j * (BK * 128), &op.maps[op.map[tap]], bar, row0 + 64 * j, w0 + op.dw[tap], h0 + op.dh[tap], n0);
  }
}

// CG = 2: the kernel runs as clusters of two CTAs that share one 256 x BN tile (tcgen05 cta_group::2): each CTA loads its own 128
// rows of A and HALF of the B tile, CTA rank 0 issues MMAs of M = 256 that read both shared memories and write both TMEMs, each
// CTA runs the epilogue of its own 128 rows.  Per MMA flop the pair pulls 2/3 of the bytes from L2 that two independent CTAs
// would (the 128 x 256 tile of one CTA needs 96 B/clk/SM at full MMA rate, above what the L2 delivers: DESIGN.md 3.2).
template <int BN, int BK, bool A_MN, bool B_MN, int EPI = 0, int CG = 1, bool HALO = false, int EW = kEpiWarps>
__global__ void __launch_bounds__(64 + 32 * EW, 1) gemm_tcgen05_kernel(const __grid_constant__ GemmParams p) {
  using S = GemmSmem<BN, BK, A_MN, B_MN, EPI, CG, HALO, EW>;
  static_assert(EW == 8 || (EW == 16 && EPI >= 1), "16 epilogue warps: linear-layer / 1x1-convolution epilogues only");
  constexpr int STAGES = S::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::BAR_OFF);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* ah_full = tmem_empty + 2;                   // HALO: ring of A halo boxes
  uint64_t* ah_empty = ah_full + kHaloStages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(ah_empty + kHaloStages);
  uint8_t* ah_smem = smem + S::AH_OFF;
  uint8_t* epi_stage = smem + S::EPI_OFF;                                         // per-warp staging tiles of the epilogue

  const uint32_t warp = warp_id();
  const uint32_t lane = lane_id();
  // tile = (row block [pair], column block, split); a CTA pair walks the same tile sequence, CTA rank r takes row block 2 * pm + r
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
  const int total_tiles = (CG == 2 ? (p.m_blocks + 1) / 2 : p.m_blocks) * p.n_blocks * p.splits;
  const int tile_first = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  // PATCH_MN stages contain rows no TMA box ever writes (K padding) -> must be zero, not garbage.
  if (p.a.mode == OP_PATCH_MN || p.b.mode == OP_PATCH_MN) {
    uint4 z = make_uint4(0, 0, 0, 0);
    for (int i = threadIdx.x; i < STAGES * S::STAGE_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = z;
    fence_proxy_async_smem();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.a.maps[0]);
    tma_prefetch_desc(&p.b.maps[0]);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < kHaloStages; ++i) {
      mbar_init(&ah_full[i], 1);
      mbar_init(&ah_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], EW * CG);   // pair: the issuing CTA waits for the epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if constexpr (CG == 2) tmem_alloc_pair(tmem_ptr, S::TMEM_COLS);
    else tmem_alloc(tmem_ptr, S::TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();     // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // Role loops are warp-uniform (all 32 lanes run the control flow and the barrier waits); only the TMA / tcgen05 issue is
  // predicated on elect.sync.  With `if (lane == 0)` around the whole loop the operands are per-thread values and ptxas wraps
  // every UTCHMMA / UTMALDG in an ELECT + R2UR.BROADCAST waterfall loop (~200 cycles per MMA issue on the critical path).
  if (warp == 0) {
    {
      // ================= TMA producer =================
      int stage = 0;
      uint32_t phase = 0;
      int ah_stage = 0;
      uint32_t ah_phase = 0;
      auto produce_residual = [&](int m_blk, int n_blk) {
        for (int r = 0; r < p.res_iters; ++r) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * S::STAGE_BYTES;
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(S::A_BYTES + S::B_BYTES));
            tma_load_2d(sa, &p.eye_map, &full_bar[stage], r * 64, 0);
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_2d(sa + S::A_BYTES + j * (64 * 128), &p.res_map, &full_bar[stage], n_blk * BN + 64 * j, m_blk * 128 + r * 64);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      };
      for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
        int split = tile % p.splits;
        int rest = tile / p.splits;
        int n_blk = rest % p.n_blocks;
        int m_blk = (rest / p.n_blocks) * CG + (int)cta_rank;
        if (EPI >= 1 && p.tile_prefetch && elect_one())
          asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(&p.tile_map)),
                       "r"(n_blk * BN), "r"(m_blk * 128)
                       : "memory");
        int k_begin = (int)(((long long)split * p.k_iters) / p.splits);
        int k_end = (int)(((long long)(split + 1) * p.k_iters) / p.splits);
        int b_row0 = n_blk * BN, b_tap = 0;
        if (p.n_blocks_per_tap > 0) {
          b_tap = n_blk / p.n_blocks_per_tap;
          b_row0 = (n_blk - b_tap * p.n_blocks_per_tap) * BN;
        }
        if constexpr (CG == 2) b_row0 += (int)cta_rank * (BN / 2);      // this CTA's half of the B tile
        // bytes one stage receives: in a pair both CTAs' loads are counted on the barrier of CTA 0, which alone posts the expectation
        const uint32_t tx = (uint32_t)(p.a.tx_bytes + p.b.tx_bytes) * CG;
        const bool post_tx = CG == 1 || cta_rank == 0;
        if constexpr (HALO) {
          // K order: channel chunk outer, filter tap inner.  One halo box per chunk (A ring), one weight tile per (chunk, tap)
          // (the pipeline stages hold B only).  The weights' K index is (tap * cchunks + chunk) * 64.
          int n0, h0, w0;
          decode_patch(p.geom, m_blk, n0, h0, w0);
          const uint32_t ah_tx = (uint32_t)(kHaloRows * 128) * CG;
          const uint32_t b_tx = (uint32_t)p.b.tx_bytes * CG;
          for (int cc = 0; cc < p.a.cchunks; ++cc) {
            mbar_wait(&ah_empty[ah_stage], ah_phase ^ 1);
            if (elect_one()) {
              if (post_tx) mbar_arrive_expect_tx(&ah_full[ah_stage], ah_tx);
              tma4<CG>(ah_smem + ah_stage * kHaloBytes, &p.a.maps[0], &ah_full[ah_stage], cc * 64, w0 + p.halo_dw0, h0 + p.halo_dh0, n0);
            }
            __syncwarp();
            if (++ah_stage == kHaloStages) { ah_stage = 0; ah_phase ^= 1; }
            for (int tap = 0; tap < p.a.ntaps; ++tap) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * S::STAGE_BYTES;
              if (elect_one()) {
                if (post_tx) mbar_arrive_expect_tx(&full_bar[stage], b_tx);
                tma2<CG>(sa, &p.b.maps[0], &full_bar[stage], (tap * p.a.cchunks + cc) * BK, b_row0);
              }
              __syncwarp();
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
          }
        } else if (p.a.mode == OP_PATCH_K && p.b.mode == OP_MAT_K) {
          // implicit-GEMM convolution fast path: patch decoded once per tile, (tap, chunk) advanced with counters —
          // this single thread's instruction latency is on the critical path of every pipeline stage
          int n0, h0, w0;
          decode_patch(p.geom, m_blk, n0, h0, w0);
          int tap = k_begin / p.a.cchunks, cc = k_begin - tap * p.a.cchunks;
          for (int kit = k_begin; kit < k_end; ++kit) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * S::STAGE_BYTES;
            if (elect_one()) {
              if (post_tx) mbar_arrive_expect_tx(&full_bar[stage], tx);
              tma4<CG>(sa, &p.a.maps[p.a.map[tap]], &full_bar[stage], cc * 64, w0 + p.a.dw[tap], h0 + p.a.dh[tap], n0);
              tma2<CG>(sa + S::A_BYTES, &p.b.maps[0], &full_bar[stage], kit * BK, b_row0);
            }
            __syncwarp();
            if (++cc == p.a.cchunks) { cc = 0; ++tap; }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        } else if (p.a.mode == OP_MAT_K && p.b.mode == OP_MAT_K) {
          for (int kit = k_begin; kit < k_end; ++kit) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * S::STAGE_BYTES;
            if (elect_one()) {
              if (post_tx) mbar_arrive_expect_tx(&full_bar[stage], tx);
              tma2<CG>(sa, &p.a.maps[0], &full_bar[stage], kit * BK, m_blk * 128);
              tma2<CG>(sa + S::A_BYTES, &p.b.maps[0], &full_bar[stage], kit * BK, b_row0);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        } else {
          for (int kit = k_begin; kit < k_end; ++kit) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * S::STAGE_BYTES;
            uint8_t* sb = sa + S::A_BYTES;
            if (elect_one()) {
              if (post_tx) mbar_arrive_expect_tx(&full_bar[stage], tx);
              issue_operand_load<128, BK, CG>(p.a, p.geom, sa, &full_bar[stage], m_blk * 128, m_blk, 0, kit);
              issue_operand_load<BN / CG, BK, CG>(p.b, p.geom, sb, &full_bar[stage], b_row0, n_blk, b_tap, kit);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        produce_residual(m_blk, n_blk);
      }
    }
  } else if (warp == 1) {
    if (CG == 1 || cta_rank == 0) {
      // ================= MMA issuer (CTA 0 of a pair) =================
      constexpr uint32_t idesc = make_idesc_bf16(128 * CG, BN, A_MN, B_MN);
      auto mma = [](uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t accum) {
        if constexpr (CG == 2) umma_bf16_pair(d, a, b, id, accum);
        else umma_bf16(d, a, b, id, accum);
      };
      auto commit = [](uint64_t* bar) {
        if constexpr (CG == 2) umma_commit_pair(bar);
        else umma_commit(bar);
      };
      // descriptor of stage 0 / k-step 0; later stages and k-steps only add to the 14-bit start-address field
      const uint32_t smem0 = smem_u32(smem);
      const uint64_t da0 = A_MN ? make_smem_desc_sw128(smem0, BK * 128, 1024) : make_smem_desc_sw128(smem0, 16, 1024);
      const uint64_t db0 = B_MN ? make_smem_desc_sw128(smem0 + S::A_BYTES, BK * 128, 1024)
                                : make_smem_desc_sw128(smem0 + S::A_BYTES, 16, 1024);
      constexpr uint64_t kStepA = (A_MN ? 2048 : 32) >> 4, kStepB = (B_MN ? 2048 : 32) >> 4;
      constexpr uint64_t kStage = S::STAGE_BYTES >> 4;
      constexpr int KSTEPS_FULL = BK / 16;
      // residual iterations: A = identity slice (K-major), B = residual rows (MN-major, 64-column chunks 8 KB apart)
      constexpr uint32_t idesc_res = make_idesc_bf16(128, BN, false, true);
      const uint64_t da_res0 = make_smem_desc_sw128(smem0, 16, 1024);
      const uint64_t db_res0 = make_smem_desc_sw128(smem0 + S::A_BYTES, 64 * 128, 1024);
      int stage = 0;
      uint32_t phase = 0;
      int ah_stage = 0;
      uint32_t ah_phase = 0;
      int it = 0;
      for (int tile = tile_first; tile < total_tiles; tile += tile_step, ++it) {
        int split = tile % p.splits;
        int k_begin = (int)(((long long)split * p.k_iters) / p.splits);
        int k_end = (int)(((long long)(split + 1) * p.k_iters) / p.splits);
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        if constexpr (HALO) {
          const uint64_t dah0 = make_smem_desc_sw128(smem_u32(ah_smem), 16, kHaloW * 128);
          for (int cc = 0; cc < p.a.cchunks; ++cc) {
            mbar_wait(&ah_full[ah_stage], ah_phase);
            tc_fence_after();
            for (int tap = 0; tap < p.a.ntaps; ++tap) {
              mbar_wait(&full_bar[stage], phase);
              tc_fence_after();
              const int shift = (p.a.dh[tap] - p.halo_dh0) * kHaloW + (p.a.dw[tap] - p.halo_dw0);     // pixel rows into the box
              const uint64_t da = dah0 + (uint64_t)((ah_stage * kHaloBytes + shift * 128) >> 4);
              const uint64_t db = db0 + (uint64_t)stage * kStage;
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) mma(d_tmem, da + k * 2, db + k * kStepB, idesc, (cc > 0 || tap > 0 || k > 0) ? 1u : 0u);
                commit(&empty_bar[stage]);
                if (tap == p.a.ntaps - 1) {
                  commit(&ah_empty[ah_stage]);
                  if (cc == p.a.cchunks - 1) commit(&tmem_full[acc]);
                }
              }
              __syncwarp();
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (++ah_stage == kHaloStages) { ah_stage = 0; ah_phase ^= 1; }
          }
          continue;
        }
        for (int kit = k_begin; kit < k_end; ++kit) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          // K-major: +32 B per 16-element K step inside the 128 B swizzle row.
          // MN-major: +2048 B per 16 k-rows (two 8-row atoms); LBO = chunk stride (BK rows x 128 B).
          const uint64_t da = da0 + (uint64_t)stage * kStage, db = db0 + (uint64_t)stage * kStage;
          if (elect_one()) {
            if (p.k_steps == KSTEPS_FULL) {
#pragma unroll
              for (int k = 0; k < KSTEPS_FULL; ++k)
                mma(d_tmem, da + k * kStepA, db + k * kStepB, idesc, (kit > k_begin || k > 0) ? 1u : 0u);
            } else {
              for (int k = 0; k < p.k_steps; ++k)
                mma(d_tmem, da + k * kStepA, db + k * kStepB, idesc, (kit > k_begin || k > 0) ? 1u : 0u);
            }
            commit(&empty_bar[stage]);  // smem slot free (in both CTAs of a pair) once these MMAs retire
            if (kit == k_end - 1 && p.res_iters == 0) commit(&tmem_full[acc]);  // accumulator complete -> epilogue
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        for (int r = 0; r < p.res_iters; ++r) {       // D += I * R  (64 residual rows per iteration)
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = da_res0 + (uint64_t)stage * kStage, db = db_res0 + (uint64_t)stage * kStage;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, da + k * 2, db + k * 128, idesc_res, 1u);
            umma_commit(&empty_bar[stage]);
            if (r == p.res_iters - 1) umma_commit(&tmem_full[acc]);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if constexpr (EPI >= 1) {
    // ================= epilogue warps (2..9), linear layers (EPI 1) / 1x1 convolutions with BatchNorm statistics (EPI 2) =========
    // Plain row-major bf16 outputs (out / pre-activation), no statistics, alpha = 1: the same split of the accumulator as below
    // (two warps per TMEM lane quarter, alternating 32-column chunks), but each 32 x 32 box is packed into a dense swizzled
    // 2 KB tile and leaves through one TMA store (bounds are clipped by the tensor map: no row / column predicates, no address
    // arithmetic, one warp barrier instead of three per box), and nothing of the convolution epilogue's state (pixel decode,
    // per-column statistics, tap decode) is live while the activation is evaluated.  EPI 2 is the same path for the 1x1
    // convolutions: bias / ReLU only, plus the per-column sums of the stored bf16 values (BatchNorm batch statistics) read back
    // from the staging tile, accumulated in registers and folded into this CTA's partial rows like the generic epilogue does.
    const uint32_t e = warp - 2;
    const uint32_t q = warp & 3;
    const uint32_t half = e >> 2;
    const uint32_t stg0 = smem_u32(epi_stage + e * 4096);
    const uint32_t swz = (lane >> 1) & 3u;                     // SWIZZLE_64B: 16-byte slot ^= (row >> 1) & 3
    const int crow = (int)(lane >> 2), cch = (int)(lane & 3);  // row-coalesced operand copies: 8 rows x 64 B per instruction
    constexpr int HALVES = EW / 4;                                   // warps per TMEM lane quarter = stride of a warp's chunks
    constexpr int NCH = (BN / 32 + HALVES - 1) / HALVES;             // 32-column chunks per epilogue warp
    constexpr bool kReadAhead = EW <= 8;                             // 16 warps: 112 registers, the accumulator is read in place
    // at most one operand tile enters the epilogue: the gate's pre-activation (aux) or a residual that could not go through the MMA.
    // It is copied global -> shared with cp.async (no registers, issued one chunk ahead into the second 2 KB tile of this warp;
    // the producer has already pulled the whole 128 x BN operand tile into L2); without an operand both tiles alternate as
    // sources of the TMA stores.
    const __nv_bfloat16* tsrc = p.aux ? p.aux : ((p.residual && p.res_iters == 0) ? p.residual : nullptr);
    const int tmode = p.aux ? p.aux_mode : 4;                  // 1 ReLU mask, 2 GELU', 3 QuickGELU', 4 add
    const uint32_t obuf = stg0 + 2048u;
    const uint32_t nalt = tsrc ? 0u : 1u;                      // store tiles in rotation
    uint32_t nbuf = 0;
    // a box is STAGED (packed into the next free 2 KB tile) and later COMMITTED (proxy fence + TMA store): the arithmetic that
    // follows the staging (activation of the saved pre-activation, column statistics) runs between the two, so that the fence
    // finds the shared-memory writes already performed
    // HALO tiles (16 x 8 pixels of one image): this warp's 32 accumulator rows are the 4 x 8 pixel box at tile rows 4q .. 4q + 3, so
    // the same dense staging tile leaves through a 4-D TMA store {32 ch, 8, 4, 1} of the NHWC output — no pixel addressing
    int hal_n0 = 0, hal_h0 = 0, hal_w0 = 0;
    bool hal_row_ok = true;
    auto stage_box = [&](const float (&f)[32], int row) -> uint32_t {
      const uint32_t buf = stg0 + (nbuf & nalt) * 2048u;
      const bool zero_row = EPI == 2 && (HALO ? !hal_row_ok : row + (int)lane >= p.M);   // rows outside the tensor must not reach the statistics
      // the store that last used this tile has read it (two boxes ago when the tiles alternate)
      if (lane == 0) {
        if (nalt) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      }
      __syncwarp();
#pragma unroll
      for (int j8 = 0; j8 < 4; ++j8) {
        uint4 u;
        u.x = pack_bf16x2(f[j8 * 8 + 0], f[j8 * 8 + 1]);
        u.y = pack_bf16x2(f[j8 * 8 + 2], f[j8 * 8 + 3]);
        u.z = pack_bf16x2(f[j8 * 8 + 4], f[j8 * 8 + 5]);
        u.w = pack_bf16x2(f[j8 * 8 + 6], f[j8 * 8 + 7]);
        if (zero_row) u = make_uint4(0u, 0u, 0u, 0u);
        st_shared_v4(buf + lane * 64u + ((j8 ^ swz) << 4), u);
      }
      ++nbuf;
      return buf;
    };
    auto commit_box = [&](uint32_t buf, const CUtensorMap* map, int col, int row) {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if constexpr (HALO)
          asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];" ::"l"(reinterpret_cast<uint64_t>(map)),
                       "r"(col), "r"(hal_w0), "r"(hal_h0 + (int)q * 4), "r"(hal_n0), "r"(buf)
                       : "memory");
        else
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(reinterpret_cast<uint64_t>(map)),
                       "r"(col), "r"(row), "r"(buf)
                       : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    };
    // EPI 2: per-warp register accumulators of the column sums (lanes 0..15 own the column pairs of each of the warp's chunks)
    float sacc[EPI == 2 ? NCH : 1][4];
#pragma unroll
    for (int i = 0; i < (EPI == 2 ? NCH : 1); ++i) { sacc[i][0] = 0.f; sacc[i][1] = 0.f; sacc[i][2] = 0.f; sacc[i][3] = 0.f; }
    auto flush_stats = [&](int nblk_) {
      if constexpr (EPI == 2) {
        float* part = p.col_sum + ((size_t)blockIdx.x * 4 + q) * 2 * p.N;
        if (lane < 16) {
#pragma unroll
          for (int i = 0; i < NCH; ++i) {
            const int col = nblk_ * BN + ((int)half + HALVES * i) * 32 + (int)lane * 2;
            if (col < p.N) {
              part[col] += sacc[i][0]; part[col + 1] += sacc[i][1];
              part[p.N + col] += sacc[i][2]; part[p.N + col + 1] += sacc[i][3];
            }
          }
        }
#pragma unroll
        for (int i = 0; i < NCH; ++i) { sacc[i][0] = 0.f; sacc[i][1] = 0.f; sacc[i][2] = 0.f; sacc[i][3] = 0.f; }
      }
    };
    int prev_nblk = -1;
    int it = 0;
    for (int tile = tile_first; tile < total_tiles; tile += tile_step, ++it) {
      const int rest = tile / p.splits;
      const int n_blk = rest % p.n_blocks;
      const int m_blk = (rest / p.n_blocks) * CG + (int)cta_rank;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int row0 = m_blk * 128 + (int)q * 32;
      const int col0 = n_blk * BN;
      if constexpr (HALO) {
        decode_patch(p.geom, m_blk, hal_n0, hal_h0, hal_w0);
        const int r_ = (int)q * 32 + (int)lane;
        hal_row_ok = hal_n0 < p.geom.Nimg && hal_h0 + (r_ >> 3) < p.geom.Ho && hal_w0 + (r_ & 7) < p.geom.Wo;
      }
      if (EPI == 2 && n_blk != prev_nblk) {
        if (prev_nblk >= 0) flush_stats(prev_nblk);
        prev_nblk = n_blk;
      }
      auto copy_tile = [&](int c_) {      // chunk c_ of the operand -> obuf (zero fill outside the tensor); one cp.async group
        const int col = col0 + c_ * 32 + cch * 8;
        const bool okc = (c_ < BN / 32) && (col < p.N);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t r_ = (uint32_t)(i * 8 + crow);
          const int m = row0 + (int)r_;
          const bool ok = okc && m < p.M;
          const __nv_bfloat16* src = ok ? tsrc + (long long)m * p.ldc + col : tsrc;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(obuf + r_ * 64u + (((uint32_t)cch ^ ((r_ >> 1) & 3u)) << 4)),
                       "l"(src), "r"(ok ? 16 : 0)
                       : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      if (tsrc) copy_tile((int)half);
      bool released = false;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((q * 32u) << 16) + acc * BN;
      // the accumulator is read one chunk ahead of the arithmetic
      uint32_t v[32];
      if (kReadAhead && (int)half < BN / 32 && col0 + (int)half * 32 < p.N) tmem_ld_32x32(t_addr + half * 32, v);
#pragma unroll 1
      for (int ci = 0; ci < NCH; ++ci) {
        const int c = (int)half + HALVES * ci;
        if (c >= BN / 32) break;
        const int cc0 = col0 + c * 32;
        if (cc0 >= p.N) break;
        if constexpr (!kReadAhead) tmem_ld_32x32(t_addr + c * 32, v);
        float4 bv[8];
        if (kReadAhead && p.bias) {
          if (cc0 + 32 <= p.N) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) bv[j4] = __ldg(reinterpret_cast<const float4*>(p.bias + cc0) + j4);
          } else {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              bv[j4] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (cc0 + j4 * 4 < p.N) bv[j4] = __ldg(reinterpret_cast<const float4*>(p.bias + cc0) + j4);   // N % 8 == 0
            }
          }
        }
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        const bool more = ci + 1 < NCH && c + HALVES < BN / 32 && cc0 + 32 * HALVES < p.N;
        if (more) {
          if constexpr (kReadAhead) tmem_ld_32x32(t_addr + (c + HALVES) * 32, v);
        } else {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]); }
          released = true;
        }
        if (p.bias) {
          if constexpr (kReadAhead) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              f[j4 * 4 + 0] += bv[j4].x; f[j4 * 4 + 1] += bv[j4].y; f[j4 * 4 + 2] += bv[j4].z; f[j4 * 4 + 3] += bv[j4].w;
            }
          } else {            // L1-resident broadcast loads, consumed four values at a time (N % 8 == 0)
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              if (cc0 + j4 * 4 < p.N) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + cc0) + j4);
                f[j4 * 4 + 0] += b4.x; f[j4 * 4 + 1] += b4.y; f[j4 * 4 + 2] += b4.z; f[j4 * 4 + 3] += b4.w;
              }
            }
          }
        }
        uint32_t pbuf = 0;
        if (EPI == 1 && p.preact) pbuf = stage_box(f, row0);
        if (p.act == ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
        } else if (EPI == 1 && p.act == ACT_GELU) {
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) act_gelu8(f + j8 * 8);
        } else if (EPI == 1 && p.act == ACT_QUICKGELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = act_quickgelu(f[j]);
        }
        if (EPI == 1 && p.preact) commit_box(pbuf, &p.pre_map, cc0, row0);
        if (tsrc) {
          asm volatile("cp.async.wait_group 0;" ::: "memory");
          __syncwarp();
          if (tmode == 1) {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<1>(f + j8 * 8, ld_shared_v4(obuf + lane * 64u + ((j8 ^ swz) << 4)));
          } else if (EPI == 1 && tmode == 2) {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<2>(f + j8 * 8, ld_shared_v4(obuf + lane * 64u + ((j8 ^ swz) << 4)));
          } else if (EPI == 1 && tmode == 3) {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<3>(f + j8 * 8, ld_shared_v4(obuf + lane * 64u + ((j8 ^ swz) << 4)));
          } else {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<4>(f + j8 * 8, ld_shared_v4(obuf + lane * 64u + ((j8 ^ swz) << 4)));
          }
          __syncwarp();
          if (ci + 1 < NCH) copy_tile(c + HALVES);       // the tile is free again: next chunk's operand
        }
        const uint32_t sbuf = stage_box(f, row0);
        if constexpr (EPI == 2) {
          __syncwarp();
          // column sums of the bf16 values just staged: lane = (row parity, column pair), 16 rows x one 32-bit word each; the
          // two lanes of a column pair are folded with one shuffle round (the TMA store reads the tile concurrently)
          // (row 2 rr + rpar sits at rr * 128 + rpar * 64; its 16-byte slots are permuted by rr & 3: four lane addresses, then
          // immediate offsets only; two independent partial sums per accumulator halve the dependent chains)
          const uint32_t wsel = lane & 15u, rpar = lane >> 4;
          const uint32_t a0 = sbuf + rpar * 64u + (wsel & 3u) * 4u;
          uint32_t ak[4];
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) ak[k] = a0 + (((wsel >> 2) ^ k) << 4);
          float sa = 0.f, sb = 0.f, qa = 0.f, qb = 0.f, sa2 = 0.f, sb2 = 0.f, qa2 = 0.f, qb2 = 0.f;
#pragma unroll
          for (int rr_ = 0; rr_ < 16; rr_ += 2) {
            const uint32_t wv = ld_shared_u32(ak[rr_ & 3] + (uint32_t)rr_ * 128u);
            const uint32_t wv2 = ld_shared_u32(ak[(rr_ + 1) & 3] + (uint32_t)(rr_ + 1) * 128u);
            const float x0 = __uint_as_float(wv << 16), x1 = __uint_as_float(wv & 0xffff0000u);
            const float y0 = __uint_as_float(wv2 << 16), y1 = __uint_as_float(wv2 & 0xffff0000u);
            sa += x0; sb += x1; sa2 += y0; sb2 += y1;
            qa = fmaf(x0, x0, qa); qb = fmaf(x1, x1, qb); qa2 = fmaf(y0, y0, qa2); qb2 = fmaf(y1, y1, qb2);
          }
          sa += sa2; sb += sb2; qa += qa2; qb += qb2;
          sa += __shfl_xor_sync(0xffffffffu, sa, 16); sb += __shfl_xor_sync(0xffffffffu, sb, 16);
          qa += __shfl_xor_sync(0xffffffffu, qa, 16); qb += __shfl_xor_sync(0xffffffffu, qb, 16);
#pragma unroll
          for (int i = 0; i < NCH; ++i)
            if (i == ci) { sacc[i][0] += sa; sacc[i][1] += sb; sacc[i][2] += qa; sacc[i][3] += qb; }
        }
        commit_box(sbuf, &p.out_map, cc0, row0);
      }
      if (!released) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]); }
      }
      if (tsrc) asm volatile("cp.async.wait_group 0;" ::: "memory");   // (a zero-fill group of a chunk beyond the tensor)
    }
    if (EPI == 2 && prev_nblk >= 0) flush_stats(prev_nblk);
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the staging tiles must outlive their stores
    __syncwarp();
  } else {
    // ================= epilogue warps (2..9) =================
    // Eight warps: warp w may only touch TMEM lanes 32*(w%4).., so two warps share each lane quarter and split the 32-column
    // chunks of the accumulator between them (chunk & 1 == half).  bf16 outputs are staged through a padded per-warp smem
    // tile so that global stores (and residual loads) are row-coalesced 64 B segments issued 8 rows per instruction instead
    // of 32 different rows per instruction — the epilogue of the K-small 1x1 convolutions is LSU-wavefront bound otherwise.
    const uint32_t e = warp - 2;
    const uint32_t q = warp & 3;
    const uint32_t half = e >> 2;
    uint8_t* stg = epi_stage + e * (32 * kEpiStride);
    const uint32_t bias_u32 = smem_u32(epi_stage + EW * 32 * kEpiStride + e * (4 * 32 * 4));
    const uint32_t stg_u32 = smem_u32(stg);
    const bool staged = !p.out_fp32;
    const bool do_stats = staged && p.col_sum != nullptr;
    // BatchNorm statistics: per-warp register accumulators (lanes 0..15 own the column pairs of each of the warp's chunks), kept
    // across tiles while the CTA stays on one column block and folded into the warp's own global partial row (row = CTA*4 + lane
    // quarter; the two warps of a quarter own disjoint columns) — no atomics, no barriers
    constexpr int NCH = (BN / 64) > 0 ? (BN / 64) : 1;        // 32-column chunks per epilogue warp
    float sacc[NCH][4];
#pragma unroll
    for (int i = 0; i < NCH; ++i) { sacc[i][0] = 0.f; sacc[i][1] = 0.f; sacc[i][2] = 0.f; sacc[i][3] = 0.f; }
    auto flush_stats = [&](int nblk_) {
      float* part = p.col_sum + ((size_t)blockIdx.x * 4 + q) * 2 * p.N;
      if (lane < 16) {
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int col = nblk_ * BN + ((int)half + 2 * i) * 32 + (int)lane * 2;
          if (col < p.N) {
            part[col] += sacc[i][0]; part[col + 1] += sacc[i][1];
            part[p.N + col] += sacc[i][2]; part[p.N + col + 1] += sacc[i][3];
          }
        }
      }
#pragma unroll
      for (int i = 0; i < NCH; ++i) { sacc[i][0] = 0.f; sacc[i][1] = 0.f; sacc[i][2] = 0.f; sacc[i][3] = 0.f; }
    };
    int prev_nblk = -1;
    int it = 0;
    for (int tile = tile_first; tile < total_tiles; tile += tile_step, ++it) {
      int rest = tile / p.splits;
      int n_blk = rest % p.n_blocks;
      int m_blk = (rest / p.n_blocks) * CG + (int)cta_rank;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;

      // row handled by this thread
      const int r = q * 32 + lane;
      bool row_ok;
      long long row_off;   // element offset of the row start in out / residual
      if (p.out_pixel) {
        int n0, h0, w0;
        decode_patch(p.geom, m_blk, n0, h0, w0);
        int tw = r % p.geom.TW;
        int t = r / p.geom.TW;
        int th = t % p.geom.TH;
        int tn = t / p.geom.TH;
        int n = n0 + tn, h = h0 + th, w = w0 + tw;
        row_ok = (tn < p.geom.TN) && (n < p.geom.Nimg) && (h < p.geom.Ho) && (w < p.geom.Wo);
        row_off = (((long long)n * p.OH + (h * p.osh + p.oh0)) * p.OW + (w * p.osw + p.ow0)) * p.ldc;
      } else {
        int m = m_blk * 128 + r;
        row_ok = m < p.M;
        row_off = (long long)m * p.ldc;
      }
      const long long row_off_pub = row_ok ? row_off : -1;   // what the other lanes see through shuffles
      int col0 = n_blk * BN;
      int col_lim = p.N;  // exclusive bound on the logical column index
      long long col_base = col0;
      if (p.n_blocks_per_tap > 0) {
        int tap = n_blk / p.n_blocks_per_tap;
        int c0 = (n_blk - tap * p.n_blocks_per_tap) * BN;
        col0 = c0;
        col_lim = p.n_per_tap;
        col_base = (long long)tap * p.n_per_tap + c0;
      }
      if (do_stats && n_blk != prev_nblk) {
        if (prev_nblk >= 0) flush_stats(prev_nblk);   // this CTA moves to another column block
        prev_nblk = n_blk;
      }

      // rows this lane touches in the row-coalesced phases (8 rows x 64 B per instruction): fetched once per tile
      const int crow = (int)(lane >> 2), cch = (int)(lane & 3);
      long long ro4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) ro4[i] = __shfl_sync(0xffffffffu, row_off_pub, i * 8 + crow);

      // residual tiles are fetched one chunk ahead with row-coalesced loads (8 rows x 64 B per instruction); the first one is
      // issued before waiting for the accumulator so that its DRAM latency hides behind the MMA
      const bool use_res = staged && p.residual != nullptr && p.res_iters == 0;
      const bool use_aux = staged && p.aux != nullptr;   // the gate's operand takes the same row-coalesced, one-chunk-ahead route
      auto load_tile = [&](const __nv_bfloat16* src, int c_, uint4 (&dst)[4]) {
        const bool okc = (c_ < BN / 32) && (col0 + c_ * 32 + cch * 8 < col_lim);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          dst[i] = make_uint4(0u, 0u, 0u, 0u);
          if (ro4[i] >= 0 && okc) dst[i] = ld_nc_v4(src + ro4[i] + col_base + c_ * 32 + cch * 8);
        }
      };
      uint4 rr[4], ar[4];
      if (use_res) load_tile(p.residual, (int)half, rr);
      if (use_aux) load_tile(p.aux, (int)half, ar);

      if (p.bias) {
        // this warp's bias slices (one per chunk) go to shared memory while the MMA is still running: the chunk loop then reads
        // them with broadcast 16-byte loads instead of waiting on global loads between the TMEM load and the arithmetic
#pragma unroll
        for (int i = 0; i < NCH && i < 4; ++i) {
          const int cb = ((int)half + 2 * i) * 32 + (int)lane;
          float bvv = 0.f;
          if (cb < BN && col0 + cb < col_lim) bvv = __ldg(p.bias + col_base + cb);
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(bias_u32 + (i * 32 + lane) * 4), "f"(bvv) : "memory");
        }
        __syncwarp();
      }
      bool released = false;

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((q * 32u) << 16) + acc * BN;
      const bool unit_alpha = p.alpha == 1.f;
#pragma unroll 1   // keep the chunk body once in the instruction stream: unrolled x4 it falls out of the instruction cache (+40 % time)
      for (int ci = 0; ci < NCH; ++ci) {
        const int c = (int)half + 2 * ci;
        if (c >= BN / 32) break;
        const int cc0 = col0 + c * 32;           // logical column of v[0] (within tap)
        const long long oc0 = col_base + c * 32; // output column of v[0]
        if (cc0 >= col_lim) break;
        uint32_t v[32];
        tmem_ld_32x32(t_addr + c * 32, v);
        const bool col_ok = cc0 + cch * 8 < col_lim;
        uint4 rn[4], an[4];
        if (use_res) load_tile(p.residual, c + 2, rn);        // next chunk of this warp
        if (use_aux) load_tile(p.aux, c + 2, an);
        tmem_ld_wait();
        float f[32];
        if (unit_alpha) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]) * p.alpha;
        }
        if (!(ci + 1 < NCH && c + 2 < BN / 32 && cc0 + 64 < col_lim)) {
          // that was this warp's last read of the accumulator: hand the TMEM buffer back before the arithmetic and the stores
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]); }
          released = true;
        }
        if (p.bias) {                               // columns outside the tensor hold 0
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const uint4 b = ld_shared_v4(bias_u32 + (ci * 32 + j4 * 4) * 4);
            f[j4 * 4 + 0] += __uint_as_float(b.x); f[j4 * 4 + 1] += __uint_as_float(b.y);
            f[j4 * 4 + 2] += __uint_as_float(b.z); f[j4 * 4 + 3] += __uint_as_float(b.w);
          }
        }
        if (p.preact) {
          if (staged) {
            // through the staging tile like the output: 8 rows x 64 B per store instruction
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              uint4 u;
              u.x = pack_bf16x2(f[j8 * 8 + 0], f[j8 * 8 + 1]);
              u.y = pack_bf16x2(f[j8 * 8 + 2], f[j8 * 8 + 3]);
              u.z = pack_bf16x2(f[j8 * 8 + 4], f[j8 * 8 + 5]);
              u.w = pack_bf16x2(f[j8 * 8 + 6], f[j8 * 8 + 7]);
              st_shared_v4(stg_u32 + lane * kEpiStride + j8 * 16, u);
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (ro4[i] >= 0 && col_ok)
                *reinterpret_cast<uint4*>(p.preact + ro4[i] + oc0 + cch * 8) = ld_shared_v4(stg_u32 + (i * 8 + crow) * kEpiStride + cch * 16);
            }
            __syncwarp();
          } else if (row_ok) {
            __nv_bfloat16* pp = p.preact + row_off + oc0;
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8)
              if (cc0 + j8 * 8 < col_lim) {
                uint4 u;
                u.x = pack_bf16x2(f[j8 * 8 + 0], f[j8 * 8 + 1]);
                u.y = pack_bf16x2(f[j8 * 8 + 2], f[j8 * 8 + 3]);
                u.z = pack_bf16x2(f[j8 * 8 + 4], f[j8 * 8 + 5]);
                u.w = pack_bf16x2(f[j8 * 8 + 6], f[j8 * 8 + 7]);
                *reinterpret_cast<uint4*>(pp + j8 * 8) = u;
              }
          }
        }
        // the activation is selected outside the element loops: each variant is its own straight-line block
        if (p.act == ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
        } else if (p.act == ACT_GELU) {
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) act_gelu8(f + j8 * 8);
        } else if (p.act == ACT_QUICKGELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = act_quickgelu(f[j]);
        }
        if (use_aux) {
#pragma unroll
          for (int i = 0; i < 4; ++i) st_shared_v4(stg_u32 + (i * 8 + crow) * kEpiStride + cch * 16, ar[i]);
          __syncwarp();
          if (p.aux_mode == 1) {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<1>(f + j8 * 8, ld_shared_v4(stg_u32 + lane * kEpiStride + j8 * 16));
          } else if (p.aux_mode == 2) {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<2>(f + j8 * 8, ld_shared_v4(stg_u32 + lane * kEpiStride + j8 * 16));
          } else {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) apply_gate8<3>(f + j8 * 8, ld_shared_v4(stg_u32 + lane * kEpiStride + j8 * 16));
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) ar[i] = an[i];
        } else if (p.aux && row_ok) {
          const __nv_bfloat16* ap = p.aux + row_off + oc0;
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            if (cc0 + j8 * 8 < col_lim) {
              const uint4 u = *reinterpret_cast<const uint4*>(ap + j8 * 8);
              if (p.aux_mode == 1) apply_gate8<1>(f + j8 * 8, u);
              else if (p.aux_mode == 2) apply_gate8<2>(f + j8 * 8, u);
              else apply_gate8<3>(f + j8 * 8, u);
            }
          }
        }
        if (!staged) {
          // fp32 outputs (split-K / wgrad accumulation, fp32 features): direct per-row path
          if (p.residual && row_ok) {
            const __nv_bfloat16* rp = p.residual + row_off + oc0;
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              if (cc0 + j8 * 8 < col_lim) {
                uint4 u = *reinterpret_cast<const uint4*>(rp + j8 * 8);
                float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
                f[j8 * 8 + 0] += a0.x; f[j8 * 8 + 1] += a0.y; f[j8 * 8 + 2] += a1.x; f[j8 * 8 + 3] += a1.y;
                f[j8 * 8 + 4] += a2.x; f[j8 * 8 + 5] += a2.y; f[j8 * 8 + 6] += a3.x; f[j8 * 8 + 7] += a3.y;
              }
            }
          }
          if (row_ok) {
            float* op = reinterpret_cast<float*>(p.out) + row_off + oc0;
            if (p.partial) {
              float* pp = p.partial + (size_t)(tile % p.splits) * p.part_stride + row_off + oc0;
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4)      // ldc % 4 == 0 (splitk path precondition): 16-byte aligned like out
                if (cc0 + j4 * 4 < col_lim)
                  *reinterpret_cast<float4*>(pp + j4 * 4) = make_float4(f[j4 * 4], f[j4 * 4 + 1], f[j4 * 4 + 2], f[j4 * 4 + 3]);
            } else if (p.atomic_add) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (cc0 + j < col_lim) red_add_f32(op + j, f[j]);
            } else {
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4)
                if (cc0 + j4 * 4 < col_lim)
                  *reinterpret_cast<float4*>(op + j4 * 4) = make_float4(f[j4 * 4], f[j4 * 4 + 1], f[j4 * 4 + 2], f[j4 * 4 + 3]);
            }
          }
          continue;
        }
        // ---- staged bf16 path ----
        if (use_res) {
#pragma unroll
          for (int i = 0; i < 4; ++i) st_shared_v4(stg_u32 + (i * 8 + crow) * kEpiStride + cch * 16, rr[i]);
          __syncwarp();
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            const uint4 u = ld_shared_v4(stg_u32 + lane * kEpiStride + j8 * 16);
            float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
            f[j8 * 8 + 0] += a0.x; f[j8 * 8 + 1] += a0.y; f[j8 * 8 + 2] += a1.x; f[j8 * 8 + 3] += a1.y;
            f[j8 * 8 + 4] += a2.x; f[j8 * 8 + 5] += a2.y; f[j8 * 8 + 6] += a3.x; f[j8 * 8 + 7] += a3.y;
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) rr[i] = rn[i];          // the tile prefetched for this warp's next chunk
        }
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8) {
          uint4 u = make_uint4(0u, 0u, 0u, 0u);                 // rows outside the tensor contribute zeros to the statistics
          if (row_ok) {
            u.x = pack_bf16x2(f[j8 * 8 + 0], f[j8 * 8 + 1]);
            u.y = pack_bf16x2(f[j8 * 8 + 2], f[j8 * 8 + 3]);
            u.z = pack_bf16x2(f[j8 * 8 + 4], f[j8 * 8 + 5]);
            u.w = pack_bf16x2(f[j8 * 8 + 6], f[j8 * 8 + 7]);
          }
          st_shared_v4(stg_u32 + lane * kEpiStride + j8 * 16, u);
        }
        __syncwarp();
        if (do_stats) {
          // per-column batch statistics of the bf16 values being stored, from the staged tile: lane = (row parity, column pair);
          // 16 rows x one 32-bit word (2 columns) each, then the two row parities are folded with one shuffle round
          const uint32_t wsel = lane & 15u, rpar = lane >> 4;
          float sa = 0.f, sb = 0.f, qa = 0.f, qb = 0.f;
#pragma unroll
          for (int rr_ = 0; rr_ < 16; ++rr_) {
            const uint32_t wv = ld_shared_u32(stg_u32 + (rr_ * 2 + rpar) * kEpiStride + wsel * 4);
            const float x0 = __uint_as_float(wv << 16), x1 = __uint_as_float(wv & 0xffff0000u);
            sa += x0; sb += x1;
            qa = fmaf(x0, x0, qa); qb = fmaf(x1, x1, qb);
          }
          sa += __shfl_xor_sync(0xffffffffu, sa, 16); sb += __shfl_xor_sync(0xffffffffu, sb, 16);
          qa += __shfl_xor_sync(0xffffffffu, qa, 16); qb += __shfl_xor_sync(0xffffffffu, qb, 16);
#pragma unroll
          for (int i = 0; i < NCH; ++i)                 // static register indexing under a rolled chunk loop
            if (i == ci) { sacc[i][0] += sa; sacc[i][1] += sb; sacc[i][2] += qa; sacc[i][3] += qb; }
        }
        __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(p.out);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (ro4[i] >= 0 && col_ok)
            *reinterpret_cast<uint4*>(outp + ro4[i] + oc0 + cch * 8) = ld_shared_v4(stg_u32 + (i * 8 + crow) * kEpiStride + cch * 16);
        }
        __syncwarp();
      }
      if (!released) {       // no chunk of this warp inside the tensor
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]); }
      }
    }
    if (do_stats && prev_nblk >= 0) flush_stats(prev_nblk);
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();     // neither CTA leaves while the other may still read its shared memory / signal its barriers
  if (warp == 1) {
    __syncwarp();
    if constexpr (CG == 2) tmem_dealloc_pair(tmem_base, S::TMEM_COLS);
    else tmem_dealloc(tmem_base, S::TMEM_COLS);
  }
}

}  // namespace pb
