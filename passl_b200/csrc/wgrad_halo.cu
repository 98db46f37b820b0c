// Stride-1 convolution weight gradient (3x3 pad 1; also the 4x1 repacked stem) with a HALO tile: one TMA load of the (8+R-1) x (16+S-1) input patch serves all
// filter taps as row-shifted views of the same SWIZZLE_128B shared-memory tile (descriptor semantics pinned by umma_probe.cu).
//
//   dw[co, r, s, ci] += sum_{n,h,w} dy[n, h, w, co] * x[n, h + r - 1, w + s - 1, ci]      (resnetimagenet.py:112-131 conv2 backward)
//
// Why: the generic implicit-GEMM wgrad (gemm.cuh, PATCH_MN) treats every tap as its own N-tile, so dy and x are re-read from L2
// nine times; at ~43-57 B/clk/SM of L2->SM bandwidth those launches run at 15 % of the tensor peak.  Here a CTA owns
// (128 output channels) x (64 input channels) x (a group of 5 or 4 taps) with one 128x64 fp32 accumulator per tap in TMEM
// (5 x 64 = 320 columns), and per 128-pixel K step moves 32 KB of dy + 23 KB of x halo for 40 (32) MMAs: ~43 B/clk.
//
//   warp 0 : TMA producer   dy box {64 co, 16, 8, 1} x 2,  x box {64 ci, 18, 10, 1}  (OOB zero fill = conv padding / ragged tiles)
//   warp 1 : MMA issuer     per tap (r, s), per tile row h: A = dy rows [16h, 16h+16) (MN-major, two 64-channel atoms),
//                           B = halo rows [(h+r)*18 + s, +16) (MN-major, start not 1024-aligned, base_offset 0)
//   warps 2..5 : epilogue   tcgen05.ld -> dw (one split) or this split's slice of the scratch that splitk_reduce adds into dw
#include "common.cuh"
#include "host_utils.h"
#include "../../include/passl_b200.h"

#include <string.h>

#include <functional>

namespace pb {

constexpr int WH_TH = 8, WH_TW = 16;                        // pixel tile (one image)
constexpr int WH_A_BYTES = 2 * 128 * 128;                   // dy: two 64-channel atoms x 128 pixels x 128 B
constexpr int WH_HALO_ROWS = (WH_TH + 2) * (WH_TW + 2);     // 180
constexpr int WH_B_BYTES = 23552;                           // 180 x 128 B rounded up to a multiple of 1024
constexpr int WH_STAGE_BYTES = WH_A_BYTES + WH_B_BYTES;     // 56320   (one 64-channel halo atom: 3 stages)
constexpr int WH_STAGES = 3;
constexpr int WH_STAGE_BYTES2 = WH_A_BYTES + 2 * WH_B_BYTES;   // 79872  (two halo atoms = 128 input channels per CTA: 2 stages)
constexpr int WH_STAGES2 = 2;
constexpr int WH_SMEM = WH_STAGES * WH_STAGE_BYTES + 256 + 1024;   // >= WH_STAGES2 * WH_STAGE_BYTES2 + 256 + 1024

struct WgradHaloParams {
  CUtensorMap dy_map, x_map;
  float* dw;
  float* partial;        // splits > 1: split s stores its sums to partial + s * Cout * R * S * Cin, reduced in split order
  int N, H, W, Cin, Cout;
  int hb, wb;            // pixel tiles per image
  int k_total;           // N * hb * wb
  int m_blocks, ci_blocks, splits;
  int R, S, pad_h, pad_w;   // filter taps (R*S <= 10) and padding: halo tile = (TH + R - 1) x (TW + S - 1) pixels
  int groups, tpg;          // tap groups per (m, ci) block and taps per group (<= 5: 5 x 64 TMEM columns)
  int halo_w, halo_rows;
  // Round 2: cib = 2 makes a CTA own 128 input channels (two halo atoms, MMA N = 128, 3 taps x 128 TMEM columns per group).  An
  // M = 128 x N = 64 MMA reads 6 KB of shared memory per 16 clk (A 4 KB + B 2 KB), three times what the SM delivers; at N = 128 it
  // is 8 KB per 32 clk — the launches with Cin >= 128 were at 0.30-0.34 of the tensor roofline on that limit.
  int cib;
};

__global__ void __launch_bounds__(192, 1) wgrad_halo_kernel(const __grid_constant__ WgradHaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int nstages = p.cib == 2 ? WH_STAGES2 : WH_STAGES;
  const int stage_bytes = p.cib == 2 ? WH_STAGE_BYTES2 : WH_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + WH_STAGES * WH_STAGE_BYTES);   // past the larger of the two rings
  uint64_t* empty_bar = full_bar + WH_STAGES;
  uint64_t* acc_full = empty_bar + WH_STAGES;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 1);
  const uint32_t warp = warp_id(), lane = lane_id();
  const int total_items = p.m_blocks * p.ci_blocks * p.groups * p.splits;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.dy_map);
    tma_prefetch_desc(&p.x_map);
    for (int i = 0; i < WH_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 4);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // work item -> (m_blk, ci_blk, tap group, split)
  auto decode = [&](int item, int& m_blk, int& ci_blk, int& grp, int& k_begin, int& k_end) {
    const int split = item % p.splits;
    int rest = item / p.splits;
    grp = rest % p.groups;
    rest /= p.groups;
    ci_blk = rest % p.ci_blocks;
    m_blk = rest / p.ci_blocks;
    k_begin = (int)(((long long)split * p.k_total) / p.splits);
    k_end = (int)(((long long)(split + 1) * p.k_total) / p.splits);
  };

  if (warp == 0) {
    // ================= TMA producer =================
    int stage = 0;
    uint32_t phase = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      int m_blk, ci_blk, grp, k_begin, k_end;
      decode(item, m_blk, ci_blk, grp, k_begin, k_end);
      const int per_img = p.hb * p.wb;
      int n = k_begin / per_img;
      int rem = k_begin - n * per_img;
      int ih = rem / p.wb, iw = rem - ih * p.wb;
      for (int kt = k_begin; kt < k_end; ++kt) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * stage_bytes;
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(WH_A_BYTES + p.cib * p.halo_rows * 128));
          const int h0 = ih * WH_TH, w0 = iw * WH_TW;
          tma_load_4d(sa, &p.dy_map, &full_bar[stage], m_blk * 128, w0, h0, n);
          tma_load_4d(sa + 128 * 128, &p.dy_map, &full_bar[stage], m_blk * 128 + 64, w0, h0, n);
          for (int a = 0; a < p.cib; ++a)
            tma_load_4d(sa + WH_A_BYTES + a * WH_B_BYTES, &p.x_map, &full_bar[stage], (ci_blk * p.cib + a) * 64, w0 - p.pad_w,
                        h0 - p.pad_h, n);
        }
        __syncwarp();
        if (++iw == p.wb) { iw = 0; if (++ih == p.hb) { ih = 0; ++n; } }
        if (++stage == nstages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t idesc = make_idesc_bf16(128, 64u * (uint32_t)p.cib, true, true);
    const uint64_t da0 = make_smem_desc_sw128(smem_u32(smem), 128 * 128, 1024);                 // LBO = next 64-channel atom
    const uint64_t db0 = make_smem_desc_sw128(smem_u32(smem + WH_A_BYTES), WH_B_BYTES, 1024);   // LBO = second halo atom (cib = 2)
    const uint32_t tap_cols = 64u * (uint32_t)p.cib;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
      int m_blk, ci_blk, grp, k_begin, k_end;
      decode(item, m_blk, ci_blk, grp, k_begin, k_end);
      const int tap0 = grp * p.tpg;
      const int ntap = (p.R * p.S - tap0) < p.tpg ? (p.R * p.S - tap0) : p.tpg;
      mbar_wait(acc_empty, (it & 1) ^ 1);      // epilogue of the previous item has drained the accumulators
      tc_fence_after();
      for (int kt = k_begin; kt < k_end; ++kt) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint64_t das = da0 + (uint64_t)((stage * stage_bytes) >> 4);
        const uint64_t dbs = db0 + (uint64_t)((stage * stage_bytes) >> 4);
        if (elect_one()) {
          for (int t = 0; t < ntap; ++t) {
            const int tap = tap0 + t;
            const int r = tap / p.S, s = tap - r * p.S;
            const uint32_t d_tmem = tmem_base + t * tap_cols;
#pragma unroll
            for (int h = 0; h < WH_TH; ++h) {
              const uint64_t da = das + (uint64_t)((h * 16 * 128) >> 4);
              const uint64_t db = dbs + (uint64_t)((((h + r) * p.halo_w + s) * 128) >> 4);
              umma_bf16(d_tmem, da, db, idesc, (kt > k_begin || h > 0) ? 1u : 0u);
            }
          }
          umma_commit(&empty_bar[stage]);
          if (kt == k_end - 1) umma_commit(acc_full);
        }
        __syncwarp();
        if (++stage == nstages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ================= epilogue warps (2..5) =================
    const uint32_t q = warp & 3;
    int it = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x, ++it) {
      int m_blk, ci_blk, grp, k_begin, k_end;
      decode(item, m_blk, ci_blk, grp, k_begin, k_end);
      const int tap0 = grp * p.tpg;
      const int ntap = (p.R * p.S - tap0) < p.tpg ? (p.R * p.S - tap0) : p.tpg;
      const int co = m_blk * 128 + (int)(q * 32 + lane);
      const bool row_ok = co < p.Cout;
      mbar_wait(acc_full, it & 1);
      tc_fence_after();
      if (k_end > k_begin) {
        for (int t = 0; t < ntap; ++t) {
          const int tap = tap0 + t;
          const int ci0 = ci_blk * 64 * p.cib;
          const size_t off = ((size_t)co * (p.R * p.S) + tap) * p.Cin + ci0;
          float* part = p.partial ? p.partial + (size_t)(item % p.splits) * p.Cout * p.R * p.S * p.Cin + off : nullptr;
          float* dst = p.dw + off;
#pragma unroll 1
          for (int c = 0; c < 2 * p.cib; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tmem_base + ((q * 32u) << 16) + t * 64 * p.cib + c * 32, v);
            tmem_ld_wait();
            if (row_ok && part) {            // Cin % 64 == 0: whole 32-channel chunks, 16-byte aligned
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4)
                *reinterpret_cast<float4*>(part + c * 32 + j4 * 4) =
                    make_float4(__uint_as_float(v[j4 * 4]), __uint_as_float(v[j4 * 4 + 1]), __uint_as_float(v[j4 * 4 + 2]),
                                __uint_as_float(v[j4 * 4 + 3]));
            } else if (row_ok) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (ci0 + c * 32 + j < p.Cin) red_add_f32(dst + c * 32 + j, __uint_as_float(v[j]));
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

int splitk_run(float* out, long long rows, long long cols, long long ld, int splits, cudaStream_t st,   // gemm_api.cu
               const std::function<int(float*)>& launch);

int g_wgrad_halo_mode = 0;   // 0 auto (size heuristic), 1 always when the shape is supported, 2 never

// returns PB_ERR_UNSUPPORTED when the shape is outside the kernel's contract (the caller then takes the generic path)
int launch_wgrad_halo(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin, int Cout, int R, int S, int pad_h,
                      int pad_w, cudaStream_t st) {
  if (g_wgrad_halo_mode == 2 || Cin % 64 || Cout % 8 || H < 12 || W < 12 || R * S > 10 || R * S < 2) return PB_ERR_UNSUPPORTED;
  WgradHaloParams p;
  memset(&p, 0, sizeof(p));
  p.dw = dw; p.N = N; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout;
  p.R = R; p.S = S; p.pad_h = pad_h; p.pad_w = pad_w;
  p.cib = Cin % 128 == 0 ? 2 : 1;
  const int tmax = p.cib == 2 ? 3 : 5;               // taps per group: 512 TMEM columns / (64 * cib)
  p.groups = (R * S + tmax - 1) / tmax;
  p.tpg = (R * S + p.groups - 1) / p.groups;
  p.halo_w = WH_TW + S - 1;
  p.halo_rows = (WH_TH + R - 1) * p.halo_w;
  if (p.halo_rows * 128 > WH_B_BYTES) return PB_ERR_UNSUPPORTED;
  p.hb = (H + WH_TH - 1) / WH_TH;
  p.wb = (W + WH_TW - 1) / WH_TW;
  p.k_total = N * p.hb * p.wb;
  p.m_blocks = (Cout + 127) / 128;
  p.ci_blocks = Cin / (64 * p.cib);
  const int base = p.m_blocks * p.ci_blocks * p.groups;
  // every work item ends with a 128 x 320 fp32 red.add epilogue: it needs a long K loop to amortise it, and the grid needs enough
  // items to fill the SMs — small batches stay on the generic kernel (measured: B=64 halo 2x slower, B=1024 halo 1.4x faster)
  int splits = (2 * num_sms() + base - 1) / base;
  const int min_iters = g_wgrad_halo_mode == 1 ? 2 : 24;
  if (splits > p.k_total / min_iters) splits = p.k_total / min_iters;
  if (splits < 1) splits = 1;
  if (g_wgrad_halo_mode != 1 && base * splits < (2 * num_sms()) / 3) return PB_ERR_UNSUPPORTED;
  p.splits = splits;
  {
    uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)W * Cout * 2, (uint64_t)H * W * Cout * 2};
    uint32_t box[4] = {64, WH_TW, WH_TH, 1};
    int rc = make_tmap_bf16(&p.dy_map, dy, 4, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
    uint32_t box[4] = {64, (uint32_t)p.halo_w, (uint32_t)(WH_TH + R - 1), 1};
    int rc = make_tmap_bf16(&p.x_map, x, 4, dims, str, box);
    if (rc) return rc;
  }
  static bool attr = false;
  if (!attr) {
    PB_CUDA_CHECK(cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WH_SMEM));
    attr = true;
  }
  const int items = base * splits;
  const int grid = items < num_sms() ? items : num_sms();
  auto launch = [&](float* partial) -> int {
    p.partial = partial;
    wgrad_halo_kernel<<<grid, 192, WH_SMEM, st>>>(p);
    PB_LAUNCH_CHECK();
    return PB_OK;
  };
  if (splits == 1) return launch(nullptr);
  return splitk_run(dw, Cout, (long long)R * S * Cin, (long long)R * S * Cin, splits, st, launch);
}

}  // namespace pb

extern "C" int passl_b200_wgrad_halo_mode(int mode) {
  if (mode < 0 || mode > 2) return pb::PB_ERR_BAD_ARG;
  pb::g_wgrad_halo_mode = mode;
  return pb::PB_OK;
}
