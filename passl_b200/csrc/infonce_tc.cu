// Fused InfoNCE forward AND backward on tcgen05 — the headline kernel (BASELINE.json: "fused InfoNCE HBM GB/s vs roofline").
//
//   logits[i, j] = scale * <Q_i, K_j>  are produced tile by tile in TMEM and consumed in place by an online
//   softmax — the [N, K] logit matrix never exists in HBM.  HBM traffic is the algorithmic minimum: the key matrix
//   (MoCo queue) is streamed exactly once by TMA, Q is read once per CTA (L2 resident).
//   SURVEY.md §8(d):  fwd bytes = (2*N*D + D*K)*2 + 4*N  (C3: 16.91 MB, 4.295 GFLOP);  bwd re-reads the keys once.
//
// Replaces: paddle.matmul(q, queue) + concat + /T + CrossEntropyLoss + topk and their autograd backward
//           (passl_v110/modeling/architectures/moco.py:178-182, heads/contrastive_head.py:37-60),
//           einsum('nc,mc->nm')/T + CE (passl/models/mocov3.py:187-198), CLIP logits + CE (clip.py:331-335).
//
// ONE launch per direction (round 1 chained three kernels: 11 of its 21 us were outside the main loop):
//   * target logits <q_i, k+_i> (or <q_i, K[label_i]>) are computed once per row by an owner CTA (row % grid), one warp per
//     row with coalesced loads, and published through an epoch-stamped flag in the persistent state buffer; every CTA picks
//     them up right before its first rank comparison;
//   * partial sums of all key slices are merged with float atomics RELATIVE to the row's own target logit
//     (sum_j 2^(y_j - y_tgt - 64) can neither vanish — the target is one of the terms — nor overflow in practice), so no
//     per-slice (max, sum) pairs have to be stored and re-read;
//   * the last CTA to take a ticket turns the sums into lse / loss / top-1 / top-5 and leaves the state zeroed.
// Main loop (per 64-key tile, per row): row max by 3-input FMNMX (also screens the rank counter: a tile whose max does not
// exceed the target, or a row whose count already reached 5, is not counted), lazy rescale against an INTEGER running max,
// and the exponentials split between MUFU.EX2 and a degree-4 polynomial on the FMA pipe (Cody-Waite with the magic-number
// rounding trick; 16 MUFU lanes/clk/SM were the round-1 bound at 0.9 us per tile).
//
// Work decomposition: CTA = (row group of MB*128 queries) x (contiguous slice of 64-key tiles).
//   warp 0 : TMA producer  (key tiles through a STAGES ring, SWIZZLE_128B)
//   warp 1 : MMA issuer    (tcgen05.mma M=128 N=64 K=16, A = Q resident in TMEM, S double-buffered;
//                           backward: + dQ[128 x D] += P[128 x 64] * Ktile[64 x D], P (bf16) written to TMEM by the softmax
//                           warps over the S columns they just read, key tile re-used from shared memory as MN-major B)
//   warps 2..2+4*MB : softmax warps (one row per thread).
#include "common.cuh"
#include "host_utils.h"
#include "../../include/passl_b200.h"

#include <string.h>

namespace pb {

constexpr int NCE_BK = 64;          // keys per tile (= MMA N)
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kRefShift = 64.f;   // slice sums are accumulated relative to 2^(target + 64): no underflow, overflow only if a
                                    // logit exceeds the target by > 130 nats (then clamped: loss finite, > 100)
constexpr float kMagic = 12582912.f;  // 1.5 * 2^23
// exponent mix of the unmasked tiles: one exponential in kPolyEvery on the FMA-pipe polynomial, the others on MUFU (C3 shape,
// us per forward: MUFU only 15.70, 1/4 15.02, 1/3 15.24, 3/8 15.25)
constexpr int kPolyEvery = 4;

struct InfoNceTcParams {
  CUtensorMap q_map;  // [N, D] bf16, box {64, 128}
  CUtensorMap k_map;  // [K, D] bf16, box {64, 64}
  const __nv_bfloat16* Q;
  const __nv_bfloat16* Kmat;
  const float* P;           // [N, D] fp32 positive keys (extra column) or null
  const long long* label;   // [N] or null
  const int* excl;          // [N] or null
  float scale, loss_scale;
  int N, K, D;
  int row_groups, slices, tiles;
  // peer-sharded keys (fused compute + collective): the key matrix is the concatenation of `shards` per-rank buffers of
  // `shard_rows` keys each, read IN PLACE over NVLink (one tensor map per rank's peer-mapped buffer); 0 = one local matrix
  int shards, shard_rows;
  unsigned peer_epoch;      // a shard is readable once my_flags[rank] >= peer_epoch (written by its owner, st.release.sys)
  const unsigned* my_flags;
  const __nv_bfloat16* shard_ptr[8];
  CUtensorMap k_maps[8];
  int tgt_mode;             // 0: owner CTA computes, epoch flags (grid <= SM count); 1: every thread computes its own row
  int poly_ok;              // exponent range allows the FMA-pipe polynomial (2.1 * scale * log2e < 120)
  // persistent state (zeroed once by the caller, left zeroed / epoch-advanced by every launch)
  unsigned* epoch; unsigned* ticket; unsigned long long* tgt_tag; float* acc_l; unsigned* acc_cnt;
  // forward outputs
  float* lse; float* tgt; float* loss_rows; float* out;
  // backward
  const float* lse_in; const float* tgt_in; const float* dloss; float* dq;
  unsigned long long* dbg;  // optional per-CTA timeline (globaltimer ns), 32 slots per CTA
};

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define NCE_STAMP(slot) do { if (p.dbg) p.dbg[blockIdx.x * 32 + (slot)] = gtime(); } while (0)
// SM cycle counter relative to the start of the CTA (globaltimer only ticks every ~256 ns)
#define NCE_STAMPC(slot) do { if (p.dbg) p.dbg[blockIdx.x * 32 + (slot)] = (unsigned long long)(clock64() - nce_c0); } while (0)

__device__ __forceinline__ float ex2_mufu(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
// 2^(a*c2 - mn) on the FMA pipe.  C = kMagic - mn with mn integer-valued, mn >= every a*c2 of the tile.
//   r = a*c2 + C rounds to C + j, j = round(a*c2); x = a*c2 - j in [-0.5, 0.5]; 2^x by a degree-4 minimax polynomial
//   (max rel. error 2.9e-6, oscillating); the exponent j - mn (<= 0, > -126 by the host's poly_ok check) is the low bits of r.
__device__ __forceinline__ float ex2_poly(float a, float c2, float C) {
  const float r = __fmaf_rn(a, c2, C);
  const float jf = __fsub_rn(r, C);
  const float x = __fmaf_rn(a, c2, -jf);
  float q = __fmaf_rn(x, 0.00958278775f, 0.0559062883f);
  q = __fmaf_rn(q, x, 0.240240991f);
  q = __fmaf_rn(q, x, 0.693124235f);
  q = __fmaf_rn(q, x, 1.0f);
  return __int_as_float(__float_as_int(q) + (__float_as_int(r) << 23));
}
// {tag, value} published / polled as ONE 64-bit word: no fences on either side (release / acquire cost a MEMBAR.GPU on the
// producer and an L1 invalidate per poll on the consumers: 27 % of all stall samples in the first version of this kernel)
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// wait (whole warp, uniform) until rank q has published its key shard for this step
__device__ __forceinline__ void nce_wait_shard(const InfoNceTcParams& p, int q) {
  unsigned v;
  const long long t0 = clock64();
  do {
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p.my_flags + q) : "memory");
    if ((int)(v - p.peer_epoch) < 0 && clock64() - t0 > 8000000000LL) {
      printf("passl_b200: peer key shard %d not published (block %d)\n", q, blockIdx.x);
      __trap();
    }
  } while ((int)(v - p.peer_epoch) < 0);
  asm volatile("fence.proxy.async.global;" ::: "memory");    // the shard is read by TMA (async proxy) next
}
// row `lab` of the (possibly sharded) key matrix
__device__ __forceinline__ const __nv_bfloat16* nce_key_row(const InfoNceTcParams& p, long long lab) {
  if (p.shards == 0) return p.Kmat + (size_t)lab * p.D;
  const int q = (int)(lab / p.shard_rows);
  return p.shard_ptr[q] + (size_t)(lab - (long long)q * p.shard_rows) * p.D;
}

// ---- shared-memory carve-up (same for forward and backward) --------------------------------------------------------------
struct NceSmem {
  uint8_t* q_smem; uint8_t* k_smem;
  uint64_t *q_ready, *k_full, *k_empty, *s_full, *s_empty, *q_full, *p_full, *dq_full, *tgt_done;
  uint32_t* tmem_ptr;
  float* tgt_s;               // [MB*128] target dot products of this CTA's rows (forward, tgt_mode 0)
  int stages, q_bytes, stage_bytes;
};
__device__ __forceinline__ NceSmem nce_carve(uint8_t* smem_raw, int MB, int D) {
  NceSmem s;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  s.q_bytes = MB * 128 * D * 2;
  s.stage_bytes = NCE_BK * D * 2;
  s.stages = (200 * 1024 - s.q_bytes) / s.stage_bytes;   // same rule as nce_plan() on the host
  if (s.stages > 8) s.stages = 8;
  s.q_smem = smem;                                       // staging only: rows go smem -> registers -> TMEM
  s.k_smem = smem + s.q_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s.k_smem + s.stages * s.stage_bytes);
  s.q_ready = bars;           // 4*MB softmax-warp arrivals: Q rows are in TMEM
  s.k_full = bars + 1;        // 8
  s.k_empty = s.k_full + 8;   // 8
  s.s_full = s.k_empty + 8;   // 2
  s.s_empty = s.s_full + 2;   // 2
  s.q_full = s.s_empty + 2;   // 1
  s.p_full = s.q_full + 1;    // 2 (backward)
  s.dq_full = s.p_full + 2;   // 1 (backward)
  s.tgt_done = s.dq_full + 1; // 1 (forward): the producer warp has collected this CTA's target logits in tgt_s
  s.tmem_ptr = reinterpret_cast<uint32_t*>(s.tgt_done + 1);
  s.tgt_s = reinterpret_cast<float*>(bars + 64);       // 512 B into the barrier block
  return s;
}

// TMA producer (whole warp 0): Q block, [forward: this CTA's share of the target logits], the first key tiles, and — once every
// softmax warp holds its target logits — the rest of the key stream.  The bulk stream saturates the SM's L2 port (~60 B/clk): in
// the first version the 8-byte target polls queued behind 112 KB of key tiles and returned ~8000 cycles late.
__device__ __forceinline__ void nce_owner_targets(const InfoNceTcParams& p, int ew, int nsw, uint32_t lane, unsigned epoch);
// ONE warp per CTA polls the tagged target words of the CTA's rows (8x fewer pollers on the same 2 KB than one poll per thread),
// parks the values in shared memory and releases the softmax warps through an mbarrier
__device__ __forceinline__ void nce_collect_targets(const InfoNceTcParams& p, const NceSmem& s, int MB, int row_base, uint32_t lane,
                                                    unsigned epoch) {
  const long long t0 = clock64();
  // all polls of a round are in flight together (a sequential loop paid one L2 round trip per 32 rows: 8 x ~700 cycles)
  constexpr int MAXG = 8;                       // up to 256 rows per CTA
  const int groups = MB * 4;
  unsigned long long w[MAXG];
  unsigned pending = 0;
#pragma unroll
  for (int g = 0; g < MAXG; ++g) {
    w[g] = 0ull;
    if (g < groups && row_base + g * 32 + (int)lane < p.N) pending |= 1u << g;
  }
  while (__any_sync(0xffffffffu, pending != 0u)) {
#pragma unroll
    for (int g = 0; g < MAXG; ++g)
      if (pending & (1u << g)) w[g] = ld_relaxed_u64(p.tgt_tag + row_base + g * 32 + lane);
#pragma unroll
    for (int g = 0; g < MAXG; ++g)
      if ((pending & (1u << g)) && (unsigned)(w[g] >> 32) == epoch + 1u) pending &= ~(1u << g);
    if (pending && clock64() - t0 > 4000000000LL) {
      printf("passl_b200: InfoNCE target flag timeout (block %d lane %d pending %x)\n", blockIdx.x, lane, pending);
      __trap();
    }
  }
#pragma unroll
  for (int g = 0; g < MAXG; ++g)
    if (g < groups) s.tgt_s[g * 32 + lane] = __uint_as_float((unsigned)w[g]);
  __syncwarp();
  if (lane == 0) mbar_arrive(s.tgt_done);
}
__device__ __forceinline__ void nce_producer(const InfoNceTcParams& p, const NceSmem& s, int MB, int row_base, int t_begin, int t_end,
                                             bool fwd, unsigned epoch, long long c0 = 0) {
  const int DC = p.D / 64;
  const uint32_t lane = lane_id();
  // the key matrix is streamed once (evict-first: it must not push the re-used operands out of L2); the query block is read
  // by every CTA of the row group (evict-last)
  const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
  if (elect_one()) {
    mbar_arrive_expect_tx(s.q_full, (uint32_t)s.q_bytes);
    for (int b = 0; b < MB; ++b)
      for (int c = 0; c < DC; ++c)
        tma_load_2d_hint(s.q_smem + (b * DC + c) * (128 * 128), &p.q_map, s.q_full, c * 64, row_base + b * 128, pol_keep);
  }
  __syncwarp();
  if (fwd) nce_owner_targets(p, 0, 1, lane, epoch);
  if (fwd && p.dbg && lane == 0) p.dbg[blockIdx.x * 32 + 30] = (unsigned long long)(clock64() - c0);
  int stage = 0;
  uint32_t phase = 0;
  int ready_shard = -1;
  for (int t = t_begin; t < t_end; ++t) {
    if (fwd && p.tgt_mode == 0 && t == t_begin + 2) nce_collect_targets(p, s, MB, row_base, lane, epoch);
    const CUtensorMap* kmap = &p.k_map;
    int krow = t * NCE_BK;
    if (p.shards) {          // tile t lives in rank q's buffer: wait for its flag once, then load straight over NVLink
      const int q = krow / p.shard_rows;
      if (q != ready_shard) { nce_wait_shard(p, q); ready_shard = q; }
      kmap = &p.k_maps[q];
      krow -= q * p.shard_rows;
    }
    mbar_wait(&s.k_empty[stage], phase ^ 1);
    if (elect_one()) {
      mbar_arrive_expect_tx(&s.k_full[stage], (uint32_t)s.stage_bytes);
      for (int c = 0; c < DC; ++c)
        tma_load_2d_hint(s.k_smem + stage * s.stage_bytes + c * (NCE_BK * 128), kmap, &s.k_full[stage], c * 64, krow, pol_stream);
    }
    __syncwarp();
    if (++stage == s.stages) { stage = 0; phase ^= 1; }
  }
  if (fwd && p.tgt_mode == 0 && t_end - t_begin <= 2) nce_collect_targets(p, s, MB, row_base, lane, epoch);
}

// softmax-warp prologue, part 1 (before anything can block): target logits of the rows this CTA owns (tgt_mode 0)
__device__ __forceinline__ void nce_owner_targets(const InfoNceTcParams& p, int ew, int nsw, uint32_t lane, unsigned epoch) {
  if (p.tgt_mode != 0) return;
  for (int row = (int)blockIdx.x + ew * (int)gridDim.x; row < p.N; row += nsw * (int)gridDim.x) {
    float acc = 0.f;
    long long lab = 0;
    if (!p.P) {
      lab = p.label[row];
      lab = lab < 0 ? 0 : (lab >= p.K ? p.K - 1 : lab);
      if (p.shards) nce_wait_shard(p, (int)(lab / p.shard_rows));
    }
    const uint64_t pol_keep = l2_policy_evict_last();
    for (int d4 = lane * 4; d4 < p.D; d4 += 128) {
      const uint2 qu = ldg_u2_hint(p.Q + (size_t)row * p.D + d4, pol_keep);
      const float2 q0 = unpack_bf16x2(qu.x), q1 = unpack_bf16x2(qu.y);
      if (p.P) {
        const float4 pa = ldg_f4_hint(p.P + (size_t)row * p.D + d4, pol_keep);
        acc += q0.x * pa.x + q0.y * pa.y + q1.x * pa.z + q1.y * pa.w;
      } else {
        const uint2 ku = __ldcv(reinterpret_cast<const uint2*>(nce_key_row(p, lab) + d4));
        const float2 k0 = unpack_bf16x2(ku.x), k1 = unpack_bf16x2(ku.y);
        acc += q0.x * k0.x + q0.y * k0.y + q1.x * k1.x + q1.y * k1.y;
      }
    }
    acc = warp_sum(acc);
    if (lane == 0)
      st_relaxed_u64(p.tgt_tag + row, ((unsigned long long)(epoch + 1u) << 32) | (unsigned long long)__float_as_uint(acc));
  }
}

// part 2: Q block smem -> registers -> TMEM (A operand of every S MMA), then arrive on q_ready
__device__ __forceinline__ void nce_stage_q(const InfoNceTcParams& p, const NceSmem& s, uint32_t tm_q, int b, uint32_t q4, uint32_t lane) {
  const int DC = p.D / 64;
  const uint32_t q_cols = p.D / 2;
  const int rl = q4 * 32 + lane;                       // row inside the 128-row block
  mbar_wait(s.q_full, 0);
  const uint32_t tq = tm_q + ((q4 * 32u) << 16) + b * q_cols;
  for (int ch = 0; ch < DC; ++ch) {
    const uint8_t* base = s.q_smem + (b * DC + ch) * (128 * 128) + (rl >> 3) * 1024 + (rl & 7) * 128;
    uint32_t w[32];
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const uint4 u = *reinterpret_cast<const uint4*>(base + (((g ^ (rl & 7)) & 7) << 4));
      w[g * 4 + 0] = u.x; w[g * 4 + 1] = u.y; w[g * 4 + 2] = u.z; w[g * 4 + 3] = u.w;
    }
    tmem_st_32x32(tq + ch * 32, w);
  }
  tmem_st_wait();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(s.q_ready);
}

// part 3 (tgt_mode 1, grids larger than the SM count): every thread computes the raw target dot product of its own row
__device__ __forceinline__ float nce_fetch_target(const InfoNceTcParams& p, int row, bool row_ok, unsigned epoch) {
  if (!row_ok) return 0.f;
  (void)epoch;
  float acc = 0.f;
  long long lab = 0;
  if (!p.P) {
    lab = p.label[row];
    lab = lab < 0 ? 0 : (lab >= p.K ? p.K - 1 : lab);
    if (p.shards) nce_wait_shard(p, (int)(lab / p.shard_rows));
  }
  for (int d = 0; d < p.D; d += 2) {
    const float2 q2 = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(p.Q + (size_t)row * p.D + d));
    if (p.P) {
      acc = fmaf(q2.x, p.P[(size_t)row * p.D + d], acc);
      acc = fmaf(q2.y, p.P[(size_t)row * p.D + d + 1], acc);
    } else {
      const float2 k2 = unpack_bf16x2(__ldcv(reinterpret_cast<const uint32_t*>(nce_key_row(p, lab) + d)));
      acc = fmaf(q2.x, k2.x, acc);
      acc = fmaf(q2.y, k2.y, acc);
    }
  }
  return acc;
}

__device__ __forceinline__ void nce_setup(const InfoNceTcParams& p, const NceSmem& s, int MB, uint32_t warp, uint32_t lane, bool bwd) {
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.q_map);
    tma_prefetch_desc(&p.k_map);
    mbar_init(s.q_ready, 4 * MB);
    mbar_init(s.q_full, 1);
    for (int i = 0; i < s.stages; ++i) {
      mbar_init(&s.k_full[i], 1);
      mbar_init(&s.k_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s.s_full[i], 1);
      mbar_init(&s.s_empty[i], 4 * MB);
      mbar_init(&s.p_full[i], 4);
    }
    mbar_init(s.dq_full, 1);
    mbar_init(s.tgt_done, 1);
    fence_barrier_init();
  }
  (void)bwd;
  if (warp == 1) tmem_alloc(s.tmem_ptr, 512);
  // programmatic dependent launch: everything above overlaps the tail of the previous kernel in the stream; nothing below
  // (global reads of Q / keys / state, global writes) may start before that kernel has completed and flushed
  asm volatile("griddepcontrol.wait;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
}

// =====================================================================================================================
// forward
// =====================================================================================================================
template <int MB>
__global__ void __launch_bounds__(64 + 128 * MB, 1) infonce_tc_fwd_kernel(const __grid_constant__ InfoNceTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ float red[3][4 * MB + 2];
  __shared__ int s_is_last;
  const NceSmem s = nce_carve(smem_raw, MB, p.D);
  const int DC = p.D / 64;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t warp = warp_id(), lane = lane_id();
  const int group = blockIdx.x / p.slices;
  const int slice = blockIdx.x - group * p.slices;
  const int row_base = group * MB * 128;
  const int t_begin = (int)((long long)slice * p.tiles / p.slices);
  const int t_end = (int)((long long)(slice + 1) * p.tiles / p.slices);
  const uint32_t q_cols = p.D / 2;                 // bf16x2 per 32-bit TMEM column

  const long long nce_c0 = clock64();
  if (threadIdx.x == 64) NCE_STAMP(0);
  nce_setup(p, s, MB, warp, lane, false);
  if (threadIdx.x == 64) NCE_STAMPC(1);
  const unsigned epoch = __ldcg(p.epoch);
  const uint32_t tmem_base = *s.tmem_ptr;
  const uint32_t tm_q = tmem_base;                       // Q (A operand): block b at columns [b*q_cols, (b+1)*q_cols)
  const uint32_t tm_s = tmem_base + MB * q_cols;         // S accumulators: (buf*MB + b) * 64

  // role loops are warp-uniform; only the TMA / tcgen05 issue is elect-predicated (keeps descriptors in uniform registers)
  if (warp == 0) {
    nce_producer(p, s, MB, row_base, t_begin, t_end, true, epoch, nce_c0);
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc = make_idesc_bf16(128, NCE_BK, false, false);
    const uint64_t db0 = make_smem_desc_sw128(smem_u32(s.k_smem), 16, 1024);   // stage 0, chunk 0, k-step 0
    mbar_wait(s.q_ready, 0);
    tc_fence_after();
    if (lane == 0) NCE_STAMPC(24);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = t_begin; t < t_end; ++t, ++it) {
      const int buf = it & 1;
      const uint32_t bphase = (it >> 1) & 1;
      mbar_wait(&s.s_empty[buf], bphase ^ 1);
      mbar_wait(&s.k_full[stage], phase);
      tc_fence_after();
      if (lane == 0 && it < 4) NCE_STAMPC(25 + it);
      const uint64_t dbs = db0 + (uint64_t)((stage * s.stage_bytes) >> 4);
      if (elect_one()) {
        for (int b = 0; b < MB; ++b) {
          const uint32_t d_tmem = tm_s + (buf * MB + b) * NCE_BK;
          const uint32_t a_tmem = tm_q + b * q_cols;
          for (int c = 0; c < DC; ++c) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts(d_tmem, a_tmem + c * 32 + k * 8, dbs + (uint64_t)((c * (NCE_BK * 128) + k * 32) >> 4), idesc,
                           (c > 0 || k > 0) ? 1u : 0u);
          }
        }
        umma_commit(&s.k_empty[stage]);
        umma_commit(&s.s_full[buf]);
      }
      __syncwarp();
      if (++stage == s.stages) { stage = 0; phase ^= 1; }
    }
  } else {
    // ---------------- softmax warps ----------------
    const int ew = warp - 2;            // 0 .. 4*MB-1
    const int b = ew >> 2;              // row block
    const uint32_t q4 = warp & 3;       // TMEM lane quarter
    const int row = row_base + b * 128 + q4 * 32 + lane;
    const bool row_ok = row < p.N;
    const float c2 = p.scale * kLog2e;  // logits in the log2 domain: y = dot * c2

    nce_stage_q(p, s, tm_q, b, q4, lane);
    if (threadIdx.x == 64) NCE_STAMPC(2);
    long long lab = -1;
    int ex = -1;
    if (row_ok) {
      if (!p.P) lab = p.label[row];
      if (p.excl) ex = p.excl[row];
    }
    float tgt_raw;
    if (p.tgt_mode == 0) {
      mbar_wait(s.tgt_done, 0);
      tgt_raw = row_ok ? s.tgt_s[b * 128 + q4 * 32 + lane] : 0.f;
    } else {
      tgt_raw = nce_fetch_target(p, row, row_ok, epoch);
      if (slice == 0 && row_ok)       // the finalizing CTA reads the targets from the state buffer
        st_relaxed_u64(p.tgt_tag + row, ((unsigned long long)(epoch + 1u) << 32) | (unsigned long long)__float_as_uint(tgt_raw));
    }
    const float tgt2 = tgt_raw * c2;
    if (threadIdx.x == 64) NCE_STAMPC(3);

    float m = -INFINITY, l = 0.f;     // m: integer-valued running max (log2 domain)
    int cnt = 0;
    int it = 0;
    for (int t = t_begin; t < t_end; ++t, ++it) {
      const int buf = it & 1;
      const uint32_t bphase = (it >> 1) & 1;
      if (threadIdx.x == 64 && it < 5) NCE_STAMPC(4 + 4 * it);
      mbar_wait(&s.s_full[buf], bphase);
      tc_fence_after();
      if (threadIdx.x == 64 && it < 5) NCE_STAMPC(5 + 4 * it);
      const uint32_t taddr = tm_s + ((q4 * 32u) << 16) + (buf * MB + b) * NCE_BK;
      uint32_t v[64];
      tmem_ld_32x32(taddr, v);
      tmem_ld_32x32(taddr + 32, v + 32);
      tmem_ld_wait();
      if (threadIdx.x == 64 && it < 5) NCE_STAMPC(6 + 4 * it);
      // TMEM buffer can be refilled as soon as the values are in registers
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.s_empty[buf]);

      const int key0 = t * NCE_BK;
      const bool special = (key0 + NCE_BK > p.K) || (ex >= key0 && ex < key0 + NCE_BK) ||
                           (lab >= key0 && lab < key0 + NCE_BK);
      if (!__any_sync(0xffffffffu, special)) {
        // fast path: everything on the raw dot products (max is monotone in the positive scale)
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int j = 0; j < 64; j += 4) {
          mx0 = max3(mx0, __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
          mx1 = max3(mx1, __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
        const float mx = fmaxf(mx0, mx1);
        // rank counter, screened: only rows that can still change (count < 5) and only tiles that contain a larger logit
        if (__any_sync(0xffffffffu, cnt < 5 && mx > tgt_raw)) {
          float c0 = 0.f, c1 = 0.f, c2n = 0.f, c3 = 0.f;
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            float g0, g1, g2, g3;
            asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(g0) : "f"(__uint_as_float(v[j])), "f"(tgt_raw));
            asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(g1) : "f"(__uint_as_float(v[j + 1])), "f"(tgt_raw));
            asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(g2) : "f"(__uint_as_float(v[j + 2])), "f"(tgt_raw));
            asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(g3) : "f"(__uint_as_float(v[j + 3])), "f"(tgt_raw));
            c0 += g0; c1 += g1; c2n += g2; c3 += g3;
          }
          cnt += (int)((c0 + c1) + (c2n + c3));
        }
        const float mn = fmaxf(m, ceilf(mx * c2));
        if (mn > m) { l *= ex2_mufu(m - mn); m = mn; }
        const float negm = -mn, C = kMagic - mn;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        if (p.poly_ok) {
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float a = __uint_as_float(v[j + u]);
              const float e = ((j + u) % kPolyEvery == 0) ? ex2_poly(a, c2, C) : ex2_mufu(fmaf(a, c2, negm));
              if (u == 0) s0 += e; else if (u == 1) s1 += e; else if (u == 2) s2 += e; else s3 += e;
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            s0 += ex2_mufu(fmaf(__uint_as_float(v[j]), c2, negm));
            s1 += ex2_mufu(fmaf(__uint_as_float(v[j + 1]), c2, negm));
            s2 += ex2_mufu(fmaf(__uint_as_float(v[j + 2]), c2, negm));
            s3 += ex2_mufu(fmaf(__uint_as_float(v[j + 3]), c2, negm));
          }
        }
        l += (s0 + s1) + (s2 + s3);
      } else {
        // tiles holding the K tail, an excluded column or the labelled column: masked, all on MUFU
        float y[64];
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const int key = key0 + j;
          const bool ok = (key < p.K) && (key != ex);
          y[j] = ok ? __uint_as_float(v[j]) * c2 : -INFINITY;
          mx = fmaxf(mx, y[j]);
          cnt += (ok && key != lab && y[j] > tgt2) ? 1 : 0;
        }
        if (mx > -INFINITY) {
          const float mn = fmaxf(m, ceilf(mx));
          float sum = 0.f;
#pragma unroll
          for (int j = 0; j < 64; ++j) sum += ex2_mufu(y[j] - mn);
          l = l * ex2_mufu(m - mn) + sum;
          m = mn;
        }
      }
      if (threadIdx.x == 64 && it < 5) { asm volatile("" :: "f"(l)); NCE_STAMPC(7 + 4 * it); }
    }
    if (row_ok) {
      // slice sum relative to 2^(target + 64); merged over the slices by float atomics (order-dependent in the last bit)
      if (m > -INFINITY) {
        const float e = fminf(m - (tgt2 + kRefShift), 100.f);
        atomicAdd(p.acc_l + row, l * ex2_mufu(e));
      }
      if (cnt > 0) atomicAdd(p.acc_cnt + row, (unsigned)(cnt < 5 ? cnt : 5));
    }
    if (threadIdx.x == 64) NCE_STAMPC(22);
    __threadfence();
    if (threadIdx.x == 64) NCE_STAMPC(23);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
  // ---------------- last CTA: sums -> lse / loss / accuracies; state back to zero ----------------
  if (threadIdx.x == 0) {
    const unsigned old = atomicInc(p.ticket, gridDim.x - 1);   // wraps back to 0 by itself
    s_is_last = (old == gridDim.x - 1);
    NCE_STAMPC(31);
  }
  __syncthreads();
  if (!s_is_last) return;
  __threadfence();
  float s_loss = 0.f, s_a1 = 0.f, s_a5 = 0.f;
  const float c2 = p.scale * kLog2e;
  for (int row = threadIdx.x; row < p.N; row += blockDim.x) {
    float L = __ldcg(p.acc_l + row);
    const unsigned cnt = __ldcg(p.acc_cnt + row);
    p.acc_l[row] = 0.f;
    p.acc_cnt[row] = 0u;
    const float tgt2 = __uint_as_float((unsigned)ld_relaxed_u64(p.tgt_tag + row)) * c2;
    if (p.P) L += 5.421010862427522e-20f;                 // the positive pair's own column: 2^(tgt - (tgt + 64))
    const float lse = (tgt2 + kRefShift + log2f(L)) * kLn2;
    const float t = tgt2 * kLn2;
    const float li = lse - t;
    p.lse[row] = lse;
    p.tgt[row] = t;
    if (p.loss_rows) p.loss_rows[row] = li;
    s_loss += li;
    s_a1 += (cnt == 0u) ? 1.f : 0.f;
    s_a5 += (cnt < 5u) ? 1.f : 0.f;
  }
  s_loss = warp_sum(s_loss); s_a1 = warp_sum(s_a1); s_a5 = warp_sum(s_a5);
  if (lane == 0) { red[0][warp] = s_loss; red[1][warp] = s_a1; red[2][warp] = s_a5; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, bb = 0.f, c = 0.f;
    for (int w = 0; w < 2 + 4 * MB; ++w) { a += red[0][w]; bb += red[1][w]; c += red[2][w]; }
    p.out[0] = p.loss_scale * a / p.N;
    p.out[1] = 100.f * bb / p.N;
    p.out[2] = 100.f * c / p.N;
    *p.epoch = epoch + 1u;
    NCE_STAMPC(29);
  }
}

// =====================================================================================================================
// backward (queries only: keys / queue / positive keys are no-grad in the reference, moco.py:162-180, mocov3.py:173-198)
//   dQ_i = scale * g * ( sum_j p_ij K_j  +  (p_i,pos - 1) k+_i   |   - K[label_i] ),   p_ij = exp(scale <q_i,K_j> - lse_i),
//   g = dloss * loss_scale / N.   P tiles are rounded to bf16 for the second MMA (fp32 accumulation in TMEM).
// =====================================================================================================================
template <int MB>
__global__ void __launch_bounds__(64 + 128 * MB, 1) infonce_tc_bwd_kernel(const __grid_constant__ InfoNceTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const NceSmem s = nce_carve(smem_raw, MB, p.D);
  const int DC = p.D / 64;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t warp = warp_id(), lane = lane_id();
  const int group = blockIdx.x / p.slices;
  const int slice = blockIdx.x - group * p.slices;
  const int row_base = group * MB * 128;
  const int t_begin = (int)((long long)slice * p.tiles / p.slices);
  const int t_end = (int)((long long)(slice + 1) * p.tiles / p.slices);
  const uint32_t q_cols = p.D / 2;

  nce_setup(p, s, MB, warp, lane, true);
  const uint32_t tmem_base = *s.tmem_ptr;
  const uint32_t tm_q = tmem_base;                        // Q: block b at [b*q_cols, ...)
  const uint32_t tm_dq = tmem_base + MB * q_cols;         // dQ accumulators: block b at b*D (fp32)
  const uint32_t tm_sp = tm_dq + MB * p.D;                // S (fp32, 64 cols) / P (bf16x2, 32 cols) per block: b*64

  if (warp == 0) {
    nce_producer(p, s, MB, row_base, t_begin, t_end, false, 0u);
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc_s = make_idesc_bf16(128, NCE_BK, false, false);
    const uint32_t idesc_pv = make_idesc_bf16(128, (uint32_t)p.D, false, true);     // B = key tile, MN-major (d contiguous)
    const uint64_t dbk0 = make_smem_desc_sw128(smem_u32(s.k_smem), 16, 1024);               // K-major view (S = Q K^T)
    const uint64_t dbm0 = make_smem_desc_sw128(smem_u32(s.k_smem), NCE_BK * 128, 1024);     // MN-major view (dQ += P K)
    mbar_wait(s.q_ready, 0);
    tc_fence_after();
    auto issue_s = [&](int b, int stage) {
      const uint64_t dbs = dbk0 + (uint64_t)((stage * s.stage_bytes) >> 4);
      const uint32_t d_tmem = tm_sp + b * NCE_BK;
      const uint32_t a_tmem = tm_q + b * q_cols;
      for (int c = 0; c < DC; ++c) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_ts(d_tmem, a_tmem + c * 32 + k * 8, dbs + (uint64_t)((c * (NCE_BK * 128) + k * 32) >> 4), idesc_s,
                       (c > 0 || k > 0) ? 1u : 0u);
      }
    };
    // first tile: S of every block
    mbar_wait(&s.k_full[0], 0);
    tc_fence_after();
    if (elect_one()) {
      for (int b = 0; b < MB; ++b) {
        issue_s(b, 0);
        umma_commit(&s.s_full[b]);
      }
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = t_begin; t < t_end; ++t, ++it) {
      int nstage = stage + 1;
      uint32_t nphase = phase;
      if (nstage == s.stages) { nstage = 0; nphase ^= 1; }
      const bool has_next = (t + 1 < t_end);
      if (has_next) mbar_wait(&s.k_full[nstage], nphase);
      for (int b = 0; b < MB; ++b) {
        mbar_wait(&s.p_full[b], it & 1);
        tc_fence_after();
        if (elect_one()) {
          // dQ_b += P_b (TMEM, 4 k-steps of 16 keys) * Ktile (MN-major: +2048 B per 16 key rows)
          const uint64_t dbm = dbm0 + (uint64_t)((stage * s.stage_bytes) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(tm_dq + b * p.D, tm_sp + b * NCE_BK + k * 8, dbm + (uint64_t)((k * 2048) >> 4), idesc_pv,
                         (it > 0 || k > 0) ? 1u : 0u);
          if (b == MB - 1) umma_commit(&s.k_empty[stage]);
          if (has_next) {
            issue_s(b, nstage);                 // in order behind the PV MMA that reads the same TMEM columns
            umma_commit(&s.s_full[b]);
          }
        }
        __syncwarp();
      }
      stage = nstage; phase = nphase;
    }
    if (elect_one()) umma_commit(s.dq_full);
    __syncwarp();
  } else {
    // ---------------- softmax warps ----------------
    const int ew = warp - 2;
    const int b = ew >> 2;
    const uint32_t q4 = warp & 3;
    const int row = row_base + b * 128 + q4 * 32 + lane;
    const bool row_ok = row < p.N;
    const float c2 = p.scale * kLog2e;

    nce_stage_q(p, s, tm_q, b, q4, lane);
    long long lab = -1;
    int ex = -1;
    float L2 = 0.f;
    if (row_ok) {
      if (!p.P) lab = p.label[row];
      if (p.excl) ex = p.excl[row];
      L2 = p.lse_in[row] * kLog2e;
    }
    const float Lc = ceilf(L2);           // integer-valued: p' = 2^(y - Lc) <= 1, true p = p' * 2^(Lc - L2)
    const float negL = -Lc, C = kMagic - Lc;
    const uint32_t taddr = tm_sp + ((q4 * 32u) << 16) + b * NCE_BK;

    int it = 0;
    for (int t = t_begin; t < t_end; ++t, ++it) {
      mbar_wait(&s.s_full[b], it & 1);
      tc_fence_after();
      uint32_t v[64];
      tmem_ld_32x32(taddr, v);
      tmem_ld_32x32(taddr + 32, v + 32);
      tmem_ld_wait();
      const int key0 = t * NCE_BK;
      const bool special = (key0 + NCE_BK > p.K) || (ex >= key0 && ex < key0 + NCE_BK);
      uint32_t w[32];
      if (!__any_sync(0xffffffffu, special)) {
        if (p.poly_ok) {
#pragma unroll
          for (int j = 0; j < 64; j += 2) {
            const float a0 = __uint_as_float(v[j]), a1 = __uint_as_float(v[j + 1]);
            const float e0 = (j % kPolyEvery == 0) ? ex2_poly(a0, c2, C) : ex2_mufu(fmaf(a0, c2, negL));
            const float e1 = ((j + 1) % kPolyEvery == 0) ? ex2_poly(a1, c2, C) : ex2_mufu(fmaf(a1, c2, negL));
            w[j >> 1] = pack_bf16x2(e0, e1);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 64; j += 2)
            w[j >> 1] = pack_bf16x2(ex2_mufu(fmaf(__uint_as_float(v[j]), c2, negL)),
                                    ex2_mufu(fmaf(__uint_as_float(v[j + 1]), c2, negL)));
        }
      } else {
#pragma unroll
        for (int j = 0; j < 64; j += 2) {
          const int k0 = key0 + j, k1 = key0 + j + 1;
          const float e0 = (k0 < p.K && k0 != ex) ? ex2_mufu(fmaf(__uint_as_float(v[j]), c2, negL)) : 0.f;
          const float e1 = (k1 < p.K && k1 != ex) ? ex2_mufu(fmaf(__uint_as_float(v[j + 1]), c2, negL)) : 0.f;
          w[j >> 1] = pack_bf16x2(e0, e1);
        }
      }
      tmem_st_32x32(taddr, w);          // P over the first 32 of the S columns this thread has just read
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.p_full[b]);
    }

    // ---------------- epilogue: dQ partial of this key slice -> global (coalesced vector reds) ----------------
    mbar_wait(s.dq_full, 0);
    tc_fence_after();
    const float g = (p.dloss ? __ldg(p.dloss) : 1.f) * p.loss_scale / (float)p.N;
    const float coef = p.scale * g;
    const float rowfac = row_ok ? coef * ex2_mufu(Lc - L2) : 0.f;
    // slice 0 also adds the term of the positive pair / the labelled column
    float extra = 0.f;
    if (slice == 0 && row_ok) extra = p.P ? coef * (__expf(p.tgt_in[row] - p.lse_in[row]) - 1.f) : -coef;
    const long long lab_c = lab < 0 ? 0 : (lab >= p.K ? p.K - 1 : lab);
    if (slice == 0 && p.shards && !p.P)
      for (int q = 0; q < p.shards; ++q) nce_wait_shard(p, q);      // the labelled rows may live in any rank's shard
    float* stg = reinterpret_cast<float*>(s.k_smem) + ew * (32 * 33);     // per-warp 32 x 32 transpose tile (ring is drained)
    const int r_sub = lane >> 3, c_sub = (lane & 7) * 4;
    for (int ch = 0; ch < p.D / 32; ++ch) {
      uint32_t v[32];
      tmem_ld_32x32(tm_dq + ((q4 * 32u) << 16) + b * p.D + ch * 32, v);
      tmem_ld_wait();
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = __uint_as_float(v[j]) * rowfac;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = i * 4 + r_sub;                       // row inside the warp's 32
        const int grow = row_base + b * 128 + q4 * 32 + rr;
        const float ex_r = __shfl_sync(0xffffffffu, extra, rr);
        const long long lab_r = __shfl_sync(0xffffffffu, lab_c, rr);
        float a0 = stg[rr * 33 + c_sub], a1 = stg[rr * 33 + c_sub + 1], a2 = stg[rr * 33 + c_sub + 2], a3 = stg[rr * 33 + c_sub + 3];
        if (grow < p.N) {
          const int col = ch * 32 + c_sub;
          if (slice == 0) {
            if (p.P) {
              const float4 pk = *reinterpret_cast<const float4*>(p.P + (size_t)grow * p.D + col);
              a0 = fmaf(ex_r, pk.x, a0); a1 = fmaf(ex_r, pk.y, a1); a2 = fmaf(ex_r, pk.z, a2); a3 = fmaf(ex_r, pk.w, a3);
            } else {
              const uint2 ku = __ldcv(reinterpret_cast<const uint2*>(nce_key_row(p, lab_r) + col));
              const float2 k0 = unpack_bf16x2(ku.x), k1 = unpack_bf16x2(ku.y);
              a0 = fmaf(ex_r, k0.x, a0); a1 = fmaf(ex_r, k0.y, a1); a2 = fmaf(ex_r, k1.x, a2); a3 = fmaf(ex_r, k1.y, a3);
            }
          }
          red_add_v4(p.dq + (size_t)grow * p.D + col, a0, a1, a2, a3);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

static void nce_plan(int N, int K, int D, int& MB, int& groups, int& slices, int& tiles, int& smem) {
  MB = (D <= 128 && N > 128) ? 2 : 1;
  if (D > 256) MB = 1;
  groups = (N + MB * 128 - 1) / (MB * 128);
  tiles = (K + NCE_BK - 1) / NCE_BK;
  slices = num_sms() / groups;
  if (slices < 1) slices = 1;
  if (slices > tiles) slices = tiles;
  int q_bytes = MB * 128 * D * 2, stage_bytes = NCE_BK * D * 2;
  int stages = (200 * 1024 - q_bytes) / stage_bytes;
  if (stages > 8) stages = 8;
  smem = q_bytes + stages * stage_bytes + 512 + 1024 + 1024;   // rings + barrier block + target staging + alignment slack
}

template <typename KernelT>
static int nce_launch(KernelT kern, const InfoNceTcParams& p, int grid, int threads, int smem, cudaStream_t st) {
  PB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));   // + static smem <= 227 KB
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  PB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, p));
  PB_LAUNCH_CHECK();
  return PB_OK;
}

struct NcePeer {            // peer-sharded key matrix (NULL pointers = single local matrix)
  const void* const* shard_ptrs; const unsigned* my_flags; int world, shard_rows; unsigned epoch;
};

static int nce_fill_params(InfoNceTcParams& p, const void* Q, const void* Kmat, const float* P, const long long* label,
                           const int* excl, float scale, float loss_scale, int N, int K, int D, int& MB, int& smem,
                           const NcePeer* peer = nullptr) {
  memset(&p, 0, sizeof(p));
  nce_plan(N, K, D, MB, p.row_groups, p.slices, p.tiles, smem);
  p.Q = reinterpret_cast<const __nv_bfloat16*>(Q);
  p.Kmat = reinterpret_cast<const __nv_bfloat16*>(Kmat);
  p.P = P; p.label = label; p.excl = excl; p.scale = scale; p.loss_scale = loss_scale; p.N = N; p.K = K; p.D = D;
  p.tgt_mode = (p.row_groups * p.slices <= num_sms()) ? 0 : 1;
  p.poly_ok = (2.1f * scale * kLog2e < 120.f) ? 1 : 0;
  uint64_t qd[2] = {(uint64_t)D, (uint64_t)N}, qs[1] = {(uint64_t)D * 2};
  uint32_t qbx[2] = {64, 128};
  int rc = make_tmap_bf16(&p.q_map, Q, 2, qd, qs, qbx);
  if (rc) return rc;
  uint32_t kbx[2] = {64, NCE_BK};
  if (peer) {
    if (peer->world < 1 || peer->world > 8 || peer->shard_rows % NCE_BK || (long long)peer->world * peer->shard_rows != K)
      return PB_ERR_BAD_ARG;
    p.shards = peer->world; p.shard_rows = peer->shard_rows; p.peer_epoch = peer->epoch; p.my_flags = peer->my_flags;
    uint64_t sd[2] = {(uint64_t)D, (uint64_t)peer->shard_rows};
    for (int q = 0; q < peer->world; ++q) {
      if (!peer->shard_ptrs[q] || (reinterpret_cast<uintptr_t>(peer->shard_ptrs[q]) & 15)) return PB_ERR_BAD_ARG;
      p.shard_ptr[q] = reinterpret_cast<const __nv_bfloat16*>(peer->shard_ptrs[q]);
      rc = make_tmap_bf16(&p.k_maps[q], peer->shard_ptrs[q], 2, sd, qs, kbx);
      if (rc) return rc;
    }
    p.k_map = p.k_maps[0];
    return PB_OK;
  }
  uint64_t kd[2] = {(uint64_t)D, (uint64_t)K};
  return make_tmap_bf16(&p.k_map, Kmat, 2, kd, qs, kbx);
}

}  // namespace pb

using namespace pb;

static unsigned long long* g_nce_dbg = nullptr;
// developer hook: per-CTA timeline buffer (uint64 [grid * 16]) filled by the next launches; NULL disables
extern "C" int passl_b200_infonce_tc_set_debug(void* buf) { g_nce_dbg = reinterpret_cast<unsigned long long*>(buf); return 0; }

// persistent state: [epoch, ticket, pad, pad][tgt_tag N x u64][acc_l N][acc_cnt N]
extern "C" long long passl_b200_infonce_tc_workspace_bytes(int N, int K, int D) {
  (void)K; (void)D;
  return 16 + (long long)N * 16;
}

// Forward.  Q [N,D] bf16 (L2-normalised queries), Kmat [K,D] bf16 keys, P [N,D] fp32 optional positive keys
// (MoCo), label int64 [N] (when P == NULL), excl int32 [N] optional.  Outputs as passl_b200_simce_fwd_f32.
// `workspace` is PERSISTENT STATE: zero-filled by the caller before its first use (and after a failed launch), one buffer
// per (N, stream); every launch leaves it ready for the next one.
static int nce_fwd_impl(const void* Q, const void* Kmat, const float* P, const long long* label, const int* excl, float scale,
                        float loss_scale, int N, int K, int D, float* lse, float* tgt, float* loss_rows, float* out_scalars,
                        void* workspace, long long workspace_bytes, void* stream, const NcePeer* peer) {
  if (N <= 0 || K <= 0 || D < 64 || D % 64 || D > 512 || !(scale > 0.f)) return PB_ERR_BAD_ARG;
  if (!P && !label) return PB_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(Q) | reinterpret_cast<uintptr_t>(Kmat) | reinterpret_cast<uintptr_t>(P)) & 15) return PB_ERR_BAD_ARG;
  if (workspace_bytes < passl_b200_infonce_tc_workspace_bytes(N, K, D)) return PB_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  InfoNceTcParams p;
  int MB, smem;
  int rc = nce_fill_params(p, Q, Kmat, P, label, excl, scale, loss_scale, N, K, D, MB, smem, peer);
  if (rc) return rc;
  unsigned* w = reinterpret_cast<unsigned*>(workspace);
  p.epoch = w; p.ticket = w + 1;
  p.tgt_tag = reinterpret_cast<unsigned long long*>(w + 4);
  p.acc_l = reinterpret_cast<float*>(w + 4 + 2 * (size_t)N);
  p.acc_cnt = w + 4 + 3 * (size_t)N;
  p.lse = lse; p.tgt = tgt; p.loss_rows = loss_rows; p.out = out_scalars;
  p.dbg = g_nce_dbg;
  const int grid = p.row_groups * p.slices, threads = 64 + 128 * MB;
  return MB == 2 ? nce_launch(infonce_tc_fwd_kernel<2>, p, grid, threads, smem, st)
                 : nce_launch(infonce_tc_fwd_kernel<1>, p, grid, threads, smem, st);
}

extern "C" int passl_b200_infonce_tc_fwd(const void* Q, const void* Kmat, const float* P, const long long* label,
                                         const int* excl, float scale, float loss_scale, int N, int K, int D, float* lse,
                                         float* tgt, float* loss_rows, float* out_scalars, void* workspace,
                                         long long workspace_bytes, void* stream) {
  return nce_fwd_impl(Q, Kmat, P, label, excl, scale, loss_scale, N, K, D, lse, tgt, loss_rows, out_scalars, workspace,
                      workspace_bytes, stream, nullptr);
}

// Fused compute + collective: the gathered-key InfoNCE of MoCo v3 / CLIP (mocov3.py:187-198: k_all = all_gather(k), labels
// arange(N) + N*rank) WITHOUT the all-gather — the key matrix is the world's `world` bf16 shards [shard_rows, D], each read in
// place from its owner's peer-mapped buffer by TMA (NVLink loads overlap the MMAs / softmax of the tiles already on chip).
// shard_ptrs: HOST array of `world` device pointers (this process's mappings, own rank included); my_flags: this rank's flag row
// (uint32[world]); a shard is consumed once my_flags[q] >= epoch (passl_b200_peer_publish_keys_bf16).  label mode only.
extern "C" int passl_b200_infonce_tc_fwd_peer(const void* Q, const void* const* shard_ptrs, const void* my_flags, int world,
                                              int shard_rows, unsigned epoch, const long long* label, const int* excl,
                                              float scale, float loss_scale, int N, int D, float* lse, float* tgt,
                                              float* loss_rows, float* out_scalars, void* workspace, long long workspace_bytes,
                                              void* stream) {
  if (!shard_ptrs || !my_flags || !label) return PB_ERR_BAD_ARG;
  NcePeer peer{shard_ptrs, reinterpret_cast<const unsigned*>(my_flags), world, shard_rows, epoch};
  return nce_fwd_impl(Q, shard_ptrs[0], nullptr, label, excl, scale, loss_scale, N, world * shard_rows, D, lse, tgt, loss_rows,
                      out_scalars, workspace, workspace_bytes, stream, &peer);
}

// Backward w.r.t. the queries.  lse / tgt: saved by the forward; dloss: device scalar (upstream grad) or NULL (= 1);
// dQ fp32 [N, D] is overwritten (zero-filled here, then accumulated over the key slices with vector reds).  D <= 256.
static int nce_bwd_impl(const void* Q, const void* Kmat, const float* P, const long long* label, const int* excl, float scale,
                        float loss_scale, int N, int K, int D, const float* lse, const float* tgt, const float* dloss, float* dQ,
                        void* stream, const NcePeer* peer) {
  if (N <= 0 || K <= 0 || D < 64 || D % 64 || D > 256 || !(scale > 0.f)) return PB_ERR_BAD_ARG;
  if (!P && !label) return PB_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(Q) | reinterpret_cast<uintptr_t>(Kmat) | reinterpret_cast<uintptr_t>(P) |
       reinterpret_cast<uintptr_t>(dQ)) & 15) return PB_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  InfoNceTcParams p;
  int MB, smem;
  int rc = nce_fill_params(p, Q, Kmat, P, label, excl, scale, loss_scale, N, K, D, MB, smem, peer);
  if (rc) return rc;
  p.lse_in = lse; p.tgt_in = tgt; p.dloss = dloss; p.dq = dQ;
  PB_CUDA_CHECK(cudaMemsetAsync(dQ, 0, (size_t)N * D * 4, st));
  const int grid = p.row_groups * p.slices, threads = 64 + 128 * MB;
  return MB == 2 ? nce_launch(infonce_tc_bwd_kernel<2>, p, grid, threads, smem, st)
                 : nce_launch(infonce_tc_bwd_kernel<1>, p, grid, threads, smem, st);
}

extern "C" int passl_b200_infonce_tc_bwd(const void* Q, const void* Kmat, const float* P, const long long* label,
                                         const int* excl, float scale, float loss_scale, int N, int K, int D,
                                         const float* lse, const float* tgt, const float* dloss, float* dQ, void* stream) {
  return nce_bwd_impl(Q, Kmat, P, label, excl, scale, loss_scale, N, K, D, lse, tgt, dloss, dQ, stream, nullptr);
}

extern "C" int passl_b200_infonce_tc_bwd_peer(const void* Q, const void* const* shard_ptrs, const void* my_flags, int world,
                                              int shard_rows, unsigned epoch, const long long* label, const int* excl,
                                              float scale, float loss_scale, int N, int D, const float* lse, const float* tgt,
                                              const float* dloss, float* dQ, void* stream) {
  if (!shard_ptrs || !my_flags || !label) return PB_ERR_BAD_ARG;
  NcePeer peer{shard_ptrs, reinterpret_cast<const unsigned*>(my_flags), world, shard_rows, epoch};
  return nce_bwd_impl(Q, shard_ptrs[0], nullptr, label, excl, scale, loss_scale, N, world * shard_rows, D, lse, tgt, dloss, dQ,
                      stream, &peer);
}
