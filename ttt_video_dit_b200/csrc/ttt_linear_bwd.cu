// TTT-Linear backward scan for sm_100a.  Replaces the Triton kernel ttt_linear_scan_backward
// (ttt/models/ssm/kernels/linear_backward.py:207-520, launched from ttt/models/ssm/linear_triton.py:203-246); the
// per-step algebra is the closed form of ttt/models/ssm/kernels/linear_backward.py:73-197 in primal variables
// (oracle/ttt_oracle.py: ttt_linear_step_backward), LayerNorm eps 1e-8.
//
// Recompute: ttt_linear_fwd_kernel<true> (trajectory mode) replays a window of the scan from a checkpoint and saves the
// bf16 operand image of the state before every step (8 KB per sequence and step + b1).  This kernel then walks the
// window backwards, ONE CTA PER (batch, head) SEQUENCE, carrying d W1^T in TMEM (fp32, rows f_out) and d b1 in smem.
//
// CS = 16 tokens is far below tcgen05's M = 128, so every token tile is stored as 4 identical copies (tile rows
// 32c + j, c = 0..3, j = token): the token-lane GEMM outputs then show each token in all four TMEM lane quadrants and the
// warps of a group split the 64 feature columns between them (16-column quarters in the K group, 32-column halves in the
// Q group; lanes 16-31 of every warp are idle).  LayerNorm row sums are exchanged between the warps of a group through
// shared memory + a named barrier.  Roles:
//   K group (warps 0-3): the sequential chain   dW' -> bf16 image -> dG = K.dW' , dK = G.dW'^T -> second-order LN
//                         backward -> dZ1 -> dK += dZ1.W1^T , dW^T += dZ1^T.K
//   Q group (warps 4-5): everything that does not depend on the carried gradient (Z1bar recompute, output-LN backward,
//                         dQ, the dZ1bar^T.Q factor tile), running up to two steps ahead.
//   issue warp (warp 6):  one thread issues every K-side MMA, folds the Q-side factor into dW^T with one K=16 MMA and
//                         refills the K / V / state-image buffers by TMA, so the compute warps never block on issue.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "bwd_common.cuh"
#include "ptx.cuh"
#include "recompute_ring.cuh"
#include "ttt_internal.h"

namespace tb {
namespace linb {

using bwd::ld_row16;
using bwd::st_global16;
using bwd::st_row16;
using bwd::warp_colsum16;

constexpr int CS = 16, F = 64, NT = 224;  // 4 K-group warps + 2 Q-group warps + 1 MMA / TMA issue warp

constexpr uint32_t SM_IMG = 0;                     // ring of 4 W1^T images (slot = step & 3), [64 f_out][64 f_in] K-major
constexpr uint32_t SM_DWI = 32768;                 // bf16 image of the carried d W1^T                             8 KB
constexpr uint32_t SM_KT = SM_DWI + 8192;          // 3 x K tile (4 copies of 16 rows)                            48 KB
constexpr uint32_t SM_QT = SM_KT + 3 * 16384;      // 3 x Q tile                                                  48 KB
constexpr uint32_t SM_G = SM_QT + 3 * 16384;       // G = -eta * gradZ1 tile                                      16 KB
constexpr uint32_t SM_DZ = SM_G + 16384;           // dZ1 tile                                                    16 KB
constexpr uint32_t SM_DZQ = SM_DZ + 16384;         // 2 x dZ1bar tile                                             32 KB
constexpr uint32_t SM_V = SM_DZQ + 2 * 16384;      // 3 x V tile [16][64]                                          6 KB
constexpr uint32_t SM_DO = SM_V + 3 * 2048;        // 3 x dOut tile [16][64]                                       6 KB
constexpr uint32_t SM_MISC = SM_DO + 3 * 2048;
constexpr uint32_t MISC_BARS = 7680;
constexpr uint32_t SM_TOTAL = SM_MISC + 8192;

constexpr uint32_t TM_DW = 0, TM_DZ = 64, TM_DG = 128, TM_DK0 = 192, TM_DK1 = 256, TM_DZQ = 320, TM_DQ = 384;

struct LinBwdParams {
  const __nv_bfloat16* last_eta;  // [BH][NC][16]
  const float *ln_w, *ln_b;       // [H][64]
  LinearImages in;                // state images of the window, two stacked sequences per record (recompute_ring.cuh)
  float *dW1, *db1;               // carried state gradient == final output: [BH][64 f_in][64 f_out], [BH][64]
  __nv_bfloat16 *dXQ, *dXK, *dXV; // [BH][NC][16][64]
  float* dEta;                    // [BH][NC][16]
  float *dlnw, *dlnb;             // [BH][64], accumulated with atomics (pre-zeroed by the host wrapper)
  int H, NC, img_slots;
  int t_hi, t_lo, t0;             // steps t_hi .. t_lo (descending); image of the state before step u = record u - t0
  int first;                      // 1: start from a zero state gradient, 0: load it from dW1 / db1
  unsigned* dbg;                  // phase-timing buffer (debug builds)
};

__device__ __forceinline__ void group_sync(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

// sum per-token partials over the 4 warps of a group: xb = [4 warps][16 tokens][4]
template <int NV>
__device__ __forceinline__ void group_rowsum(float* xb, int gw, int j, bool act, int bar_id, float* v) {
  if (act) {
#pragma unroll
    for (int n = 0; n < NV; ++n) xb[(gw * 16 + j) * 4 + n] = v[n];
  }
  group_sync(bar_id);
#pragma unroll
  for (int n = 0; n < NV; ++n) v[n] = (xb[j * 4 + n] + xb[(16 + j) * 4 + n]) + (xb[(32 + j) * 4 + n] + xb[(48 + j) * 4 + n]);
}

// the Q group is a pair of warps
__device__ __forceinline__ void pair_sync() { asm volatile("bar.sync 2, 64;" ::: "memory"); }
template <int NV>
__device__ __forceinline__ void pair_rowsum(float* xb, int gw, int j, bool act, float* v) {
  if (act) {
#pragma unroll
    for (int n = 0; n < NV; ++n) xb[(gw * 16 + j) * 4 + n] = v[n];
  }
  pair_sync();
#pragma unroll
  for (int n = 0; n < NV; ++n) v[n] = xb[j * 4 + n] + xb[(16 + j) * 4 + n];
}

// 16 fp32 -> bf16 -> the 4 copies of token row j (tile rows 32c + j), chunks chunk0, chunk0 + 1
__device__ __forceinline__ void st_tok4(uint32_t tile, int j, int chunk0, const float* v) {
  const uint32_t a0 = pack_bf16(v[0], v[1]), a1 = pack_bf16(v[2], v[3]), a2 = pack_bf16(v[4], v[5]), a3 = pack_bf16(v[6], v[7]);
  const uint32_t b0 = pack_bf16(v[8], v[9]), b1 = pack_bf16(v[10], v[11]), b2 = pack_bf16(v[12], v[13]), b3 = pack_bf16(v[14], v[15]);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    st_shared_v4(tile + sw128_off(32 * c + j, chunk0), a0, a1, a2, a3);
    st_shared_v4(tile + sw128_off(32 * c + j, chunk0 + 1), b0, b1, b2, b3);
  }
}

// single-thread MMA helpers (all outputs M = 128 lanes x N = 64 columns)
__device__ __forceinline__ void mma_kk(uint32_t d, uint32_t a_tile, uint32_t b_tile) {  // D = A[128x64] . B[64x64]^T, both K-major
  constexpr uint32_t idesc = make_idesc_bf16(128, 64, false, false);
  const uint64_t da = make_desc_sw128(a_tile, 16, 1024), db = make_desc_sw128(b_tile, 16, 1024);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_ss(d, desc_advance(da, 32 * k), desc_advance(db, 32 * k), idesc, k > 0);
}
__device__ __forceinline__ void mma_kn(uint32_t d, uint32_t a_tile, uint32_t b_tile, bool acc) {  // D (+)= A[128x64] . B[64 k][64 n] (B MN-major)
  constexpr uint32_t idesc = make_idesc_bf16(128, 64, false, true);
  const uint64_t da = make_desc_sw128(a_tile, 16, 1024), db = make_desc_sw128(b_tile, 1024, 1024);
#pragma unroll
  for (int k = 0; k < 4; ++k) umma_ss(d, desc_advance(da, 32 * k), desc_advance(db, 2048 * k), idesc, acc || k > 0);
}
// rank-16 update of the state gradient: D[f_out][f_in] += sum_tok A[tok][f_out] . B[tok][f_in] over tile rows 0-15 (copy 0
// of both tiles, MN-major).  LBO = 0 aliases the second 64-row block of A onto the first, so TMEM lanes 64-127 hold a copy
// of rows 0-63 (umma self-test mode 6) and all 128 K-group threads can convert the accumulator.
__device__ __forceinline__ void mma_upd(uint32_t d, uint32_t a_tile, uint32_t b_tile) {
  constexpr uint32_t idesc = make_idesc_bf16(128, 64, true, true);
  umma_ss(d, make_desc_sw128(a_tile, 0, 1024), make_desc_sw128(b_tile, 1024, 1024), idesc, 1);
}

// seven warps: no SM sub-partition hosts more than two, so every thread may use up to 255 registers (a ninth warp
// would put three on one sub-partition and cap the kernel at 168)
__global__ void __launch_bounds__(NT, 1)
ttt_linear_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                      const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO,
                      const LinBwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = uniform_warp_id();  // == warp, provably warp-uniform: the role dispatch and the issue warp branch on it
  const int grp = warp_u >> 2;  // 0 = K group (warps 0-3); warps 4-5 = Q group, warp 6 = issue warp
  const int gw = warp & 3;    // warp within the group = TMEM lane quadrant = 16-column quarter
  const int j = lane & 15;    // token row
  const bool act = lane < 16;
  const int c0 = 16 * gw;
  const int bh = blockIdx.x, head = bh % p.H;
  const int NC = p.NC;
  const int nst = p.t_hi - p.t_lo + 1;
  const uint32_t lane_addr = ((uint32_t)(gw * 32)) << 16;
  TICK_DECL(12, 128)

  float* fm = reinterpret_cast<float*>(smem + SM_MISC);
  float* b1s = fm;          // [4][64] b1 of the image ring
  float* qdb1 = fm + 1664;  // [4][64] column sums of dZ1bar (Q group -> K group; read by the K group AFTER the factor
                            // tile of the same step was consumed, so it needs its own, deeper ring)
  float* db1c = fm + 384;   // [64] carried d b1
  float* db1n = fm + 448;   // [64] d b1 after this step's Q side
  float* lnw = fm + 512;
  float* lnb = fm + 576;
  float* xk = fm + 640;     // [2][256] K-group row-sum exchange
  float* xq = fm + 1152;    // [2][256] Q-group row-sum exchange
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_MISC + MISC_BARS);
  uint64_t* bar_k = bars;          // [3] K, V tiles
  uint64_t* bar_q = bars + 3;      // [3] Q, dOut tiles
  uint64_t* bar_img = bars + 6;    // [4] state images (+ b1)
  uint64_t* bar_mz = bars + 10;    // Z1 recompute MMA
  uint64_t* bar_mg = bars + 11;    // dG, dK(a) MMAs
  uint64_t* bar_mkb = bars + 12;   // dK(b) + K-side state update
  uint64_t* bar_upd = bars + 13;   // state gradient complete for the next step
  uint64_t* bar_qready = bars + 14;  // [2] Q-side factor tile written
  uint64_t* bar_qfree = bars + 16;   // [2] Q-side factor tile consumed
  uint64_t* bar_mq = bars + 18;    // Q-group MMAs
  uint64_t* bar_kb = bars + 19;    // K group -> issue warp: state-gradient image + G tile written (first: TMEM state loaded)
  uint64_t* bar_ke = bars + 20;    // K group -> issue warp: dZ1 tile written
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 22);

  if (tid == 0) {
    for (int i = 0; i < 21; ++i) mbar_init(&bars[i], 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmDO);
  }
  if (warp == 0) tmem_alloc<512>(tmem_ptr);
  for (int i = tid; i < (int)(SM_MISC / 16); i += NT) st_shared_v4(sbase + 16 * i, 0, 0, 0, 0);  // idle tile rows stay 0
  if (tid < 64) {
    lnw[tid] = p.ln_w[head * F + tid];
    lnb[tid] = p.ln_b[head * F + tid];
    db1c[tid] = p.first ? 0.f : p.db1[(size_t)bh * F + tid];
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;

  const uint8_t* img_g = p.in.image(bh >> 1, p.img_slots, 0) + (size_t)(bh & 1) * kLinSeqImageBytes;
  const float* b1_g = p.in.image_b1(bh >> 1, p.img_slots, 0) + (bh & 1) * kLinSeqB1Floats;
  auto load_image = [&](int u) {  // state before step u -> ring slot u & 3
    const int s = u & 3;
    mbar_expect_tx(&bar_img[s], 8192 + 256);
    bulk_load_1d(smem + SM_IMG + s * 8192, img_g + (size_t)(u - p.t0) * kLinImageBytes, 8192, &bar_img[s]);
    bulk_load_1d(b1s + s * 64, b1_g + (size_t)(u - p.t0) * kLinImageB1Floats, 256, &bar_img[s]);
  };
  auto load_k = [&](int i) {  // K, V of step index i (t = t_hi - i) -> slot i % 3
    const int s = i % 3, row = (bh * NC + (p.t_hi - i)) * CS;
    mbar_expect_tx(&bar_k[s], 5 * 2048);
#pragma unroll
    for (int c = 0; c < 4; ++c) tma_load_2d(smem + SM_KT + s * 16384 + c * 4096, &tmK, 0, row, &bar_k[s]);
    tma_load_2d(smem + SM_V + s * 2048, &tmV, 0, row, &bar_k[s]);
  };
  auto load_q = [&](int i) {
    const int s = i % 3, row = (bh * NC + (p.t_hi - i)) * CS;
    mbar_expect_tx(&bar_q[s], 5 * 2048);
#pragma unroll
    for (int c = 0; c < 4; ++c) tma_load_2d(smem + SM_QT + s * 16384 + c * 4096, &tmQ, 0, row, &bar_q[s]);
    tma_load_2d(smem + SM_DO + s * 2048, &tmDO, 0, row, &bar_q[s]);
  };

  if (grp == 0) {
    // =============================================== K group ========================================================
    {  // carried d W1^T -> TMEM (lanes 64-127 mirror lanes 0-63)
      const int row = tid & 63;
      const float* src = p.dW1 + (size_t)bh * F * F;
      uint32_t v[32];
#pragma unroll
      for (int c = 0; c < 2; ++c) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = p.first ? 0u : __float_as_uint(src[(size_t)(32 * c + i) * F + row]);
        tmem_st32(tmem + lane_addr + TM_DW + 32 * c, v);
      }
      tc_wait_st();
    }
    tc_fence_before();
    group_sync(1);
    if (tid == 0) mbar_arrive(bar_kb);

    float eta_c = __bfloat162float(p.last_eta[((size_t)bh * NC + p.t_hi) * CS + j]);
    float dgam[16], dbet[16], dyp[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) { dgam[e] = 0.f; dbet[e] = 0.f; dyp[e] = 0.f; }
    int xsel = 0;

    for (int i = 0; i < nst; ++i) {
      const int t = p.t_hi - i;
      const int ks = i % 3;
      const uint32_t kt = sbase + SM_KT + ks * 16384, vt = sbase + SM_V + ks * 2048;
      const uint32_t gt = sbase + SM_G, dzt = sbase + SM_DZ, dwi = sbase + SM_DWI;
      const float* b1t = b1s + (t & 3) * 64;
      const float eta_n = (i + 1 < nst) ? __bfloat162float(p.last_eta[((size_t)bh * NC + t - 1) * CS + j]) : 0.f;

      // ---- (A) first-order pass of the K side: Z1 -> LayerNorm -> gradZ1 -> G = -eta * gradZ1   (independent of the carry)
      mbar_wait(&bar_k[ks], (i / 3) & 1);
      mbar_wait(&bar_img[t & 3], ((i + 1) >> 2) & 1);
      mbar_wait(bar_mz, i & 1);
      tc_fence_after();
      TICK(0);  // loop tail + waits for K/V, image, Z1 MMA
      float xh[16], gxh[16], go[16], gz[16];
      float rstd, s2c;
      {
        uint32_t r[16];
        tmem_ld16(tmem + lane_addr + TM_DZ + c0, r);
        tc_wait_ld();
        float z[16], ex[2] = {0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          z[e] = __uint_as_float(r[e]) + b1t[c0 + e];
          ex[0] += z[e];
          ex[1] = fmaf(z[e], z[e], ex[1]);
        }
        group_rowsum<2>(xk + xsel * 256, gw, j, act, 1, ex);
        xsel ^= 1;
        const float mu = ex[0] * (1.f / 64.f);
        rstd = rsqrtf(fmaxf(ex[1] * (1.f / 64.f) - mu * mu, 0.f) + 1e-8f);
        float kk[16], vv[16];
        ld_row16(kt, j, 2 * gw, kk);
        ld_row16(vt, j, 2 * gw, vv);
        float qs[2] = {0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          xh[e] = (z[e] - mu) * rstd;
          go[e] = fmaf(lnw[c0 + e], xh[e], lnb[c0 + e]) - (vv[e] - kk[e]);
          gxh[e] = go[e] * lnw[c0 + e];
          qs[0] += gxh[e];
          qs[1] = fmaf(gxh[e], xh[e], qs[1]);
        }
        group_rowsum<2>(xk + xsel * 256, gw, j, act, 1, qs);
        xsel ^= 1;
        s2c = qs[1];
        const float sc = rstd * (1.f / 64.f);
        float gv[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          gz[e] = (fmaf(64.f, gxh[e], -qs[0]) - xh[e] * s2c) * sc;
          gv[e] = -eta_c * gz[e];
        }
        if (act) st_tok4(gt, j, 2 * gw, gv);
      }

      TICK(1);  // first-order pass
      // ---- (B) carried d W1^T (complete once last step's update and this step's Q-side factor landed) -> bf16 image
      mbar_wait(bar_upd, i & 1);
      tc_fence_after();
      TICK(2);  // wait for the state gradient
      {
        const int row = tid & 63, half = tid >> 6;
        uint32_t v[32];
        tmem_ld32(tmem + lane_addr + TM_DW + 32 * half, v);
        tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 4; ++q)
          st_shared_v4(dwi + sw128_off(row, 4 * half + q),
                       pack_bf16(__uint_as_float(v[8 * q]), __uint_as_float(v[8 * q + 1])),
                       pack_bf16(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3])),
                       pack_bf16(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5])),
                       pack_bf16(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7])));
      }
      if (tid < 64) db1n[tid] = db1c[tid] + qdb1[(i & 3) * 64 + tid];
      fence_proxy_async();
      tc_fence_before();
      group_sync(1);

      TICK(3);  // accumulator -> bf16 image
      // ---- (C) issue warp: dG = K . dW1' ; dK = G . dW1'^T ; then the next step's Z1 recompute
      if (tid == 0) mbar_arrive(bar_kb);

      TICK(4);  // MMA issue
      // ---- (D) deferred epilogue of the previous step: d XK, then refill the buffers it released
      if (i > 0) {
        mbar_wait(bar_mkb, (i - 1) & 1);
        tc_fence_after();
        uint32_t r[16];
        tmem_ld16(tmem + lane_addr + (((i - 1) & 1) ? TM_DK1 : TM_DK0) + c0, r);
        tc_wait_ld();
        if (act) {
          float o[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) o[e] = __uint_as_float(r[e]) + dyp[e];
          st_global16(p.dXK + (((size_t)bh * NC + t + 1) * CS + j) * F + c0, o);
        }
      }

      TICK(5);  // deferred d XK epilogue + refills
      // ---- (E) second-order pass: backward through gradZ1 = ln_fused_l2_bwd(Z1, V - K)
      mbar_wait(bar_mg, i & 1);
      tc_fence_after();
      TICK(6);  // wait for dG
      {
        uint32_t r[16];
        tmem_ld16(tmem + lane_addr + TM_DG + c0, r);
        tc_wait_ld();
        float dgz[16], ex[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const float dG = __uint_as_float(r[e]) + db1n[c0 + e];
          dgz[e] = -eta_c * dG;
          ex[0] += dgz[e];
          ex[1] = fmaf(dgz[e], xh[e], ex[1]);
          ex[2] = fmaf(gz[e], dG, ex[2]);
        }
        group_rowsum<3>(xk + xsel * 256, gw, j, act, 1, ex);
        xsel ^= 1;
        if (gw == 0 && act) p.dEta[((size_t)bh * NC + t) * CS + j] = -ex[2];
        float dxh[16], sx[2] = {0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const float dgxh = (dgz[e] - (ex[0] + xh[e] * ex[1]) * (1.f / 64.f)) * rstd;
          const float dy = lnw[c0 + e] * dgxh;
          if (act) {
            dgam[e] += fmaf(go[e], dgxh, dy * xh[e]);
            dbet[e] += dy;
          }
          dyp[e] = dy;  // = -d target: d XV = -dy, d XK gets +dy
          dxh[e] = fmaf(dy, lnw[c0 + e], -(gxh[e] * ex[1] + dgz[e] * s2c) * rstd * (1.f / 64.f));
          sx[0] += (-dxh[e] * xh[e] - dgz[e] * gz[e]) * rstd;
          sx[1] += dxh[e];
        }
        group_rowsum<2>(xk + xsel * 256, gw, j, act, 1, sx);
        xsel ^= 1;
        float dz[16], nv[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          dz[e] = fmaf(dxh[e], rstd, (sx[0] * xh[e] - sx[1] * rstd) * (1.f / 64.f));
          nv[e] = -dyp[e];
        }
        if (act) {
          st_tok4(dzt, j, 2 * gw, dz);
          st_global16(p.dXV + (((size_t)bh * NC + t) * CS + j) * F + c0, nv);
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) dz[e] = 0.f;
        }
        warp_colsum16(dz, lane);  // d b1 += column sums of dZ1 over the 16 tokens
        if ((lane & 1) == 0) db1c[c0 + (lane >> 1)] = db1n[c0 + (lane >> 1)] + dz[0];
      }
      fence_proxy_async();
      tc_fence_before();
      group_sync(1);

      TICK(7);  // second-order pass
      // ---- (F) issue warp: dK += dZ1 . W1^T ; dW^T += dZ1^T . K ; then fold the next step's Q-side factor
      if (tid == 0) mbar_arrive(bar_ke);
      eta_c = eta_n;
      TICK(8);  // MMA issue (+ wait for the Q-side factor)
    }

    // ---- epilogue of the last step + carried state gradient -> global
    mbar_wait(bar_mkb, (nst - 1) & 1);
    tc_fence_after();
    {
      uint32_t r[16];
      tmem_ld16(tmem + lane_addr + (((nst - 1) & 1) ? TM_DK1 : TM_DK0) + c0, r);
      tc_wait_ld();
      if (act) {
        float o[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] = __uint_as_float(r[e]) + dyp[e];
        st_global16(p.dXK + (((size_t)bh * NC + p.t_lo) * CS + j) * F + c0, o);
      }
    }
    {
      const int row = tid & 63, half = tid >> 6;
      float* dst = p.dW1 + (size_t)bh * F * F;
      uint32_t v[32];
      tmem_ld32(tmem + lane_addr + TM_DW + 32 * half, v);
      tc_wait_ld();
#pragma unroll
      for (int e = 0; e < 32; ++e) dst[(size_t)(32 * half + e) * F + row] = __uint_as_float(v[e]);
    }
    group_sync(1);
    if (tid < 64) p.db1[(size_t)bh * F + tid] = db1c[tid];
    if (!act) {
#pragma unroll
      for (int e = 0; e < 16; ++e) { dgam[e] = 0.f; dbet[e] = 0.f; }
    }
    warp_colsum16(dgam, lane);
    warp_colsum16(dbet, lane);
    if ((lane & 1) == 0) {
      atomicAdd(p.dlnw + (size_t)bh * F + c0 + (lane >> 1), dgam[0]);
      atomicAdd(p.dlnb + (size_t)bh * F + c0 + (lane >> 1), dbet[0]);
    }
  } else if (warp_u < 6) {
    // =============================================== Q group ========================================================
    // two warps (TMEM lane quadrants 0 and 1), each thread = one token x 32 columns: this group has slack, and seven
    // warps in total keep every SM sub-partition at two warps, i.e. the full 255-register budget for the K group
    const int q0 = 32 * gw;  // first column of this thread
    if (tid == 128)
      for (int i = 0; i < 3 && i < nst; ++i) load_q(i);
    float dgq[32], dbq[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) { dgq[e] = 0.f; dbq[e] = 0.f; }
    uint32_t mq_phase = 0;
    int xsel = 0;
    for (int i = 0; i < nst; ++i) {
      const int t = p.t_hi - i;
      const int qs3 = i % 3, ds = i & 1;
      const uint32_t qt = sbase + SM_QT + qs3 * 16384, dot = sbase + SM_DO + qs3 * 2048;
      const uint32_t dzq = sbase + SM_DZQ + ds * 16384;
      const uint32_t img_n = sbase + SM_IMG + ((t + 1) & 3) * 8192;  // state AFTER step t
      const float* b1n = b1s + ((t + 1) & 3) * 64;

      mbar_wait(&bar_q[qs3], (i / 3) & 1);
      mbar_wait(&bar_img[(t + 1) & 3], (i >> 2) & 1);
      TICK(0);  // waits for Q/dOut, image
      if (tid == 128) {
        tc_fence_after();
        mma_kk(tmem + TM_DZQ, qt, img_n);  // Z1bar = Q . W1'
        tc_commit(bar_mq);
      }
      mbar_wait(bar_mq, mq_phase);
      mq_phase ^= 1;
      tc_fence_after();
      TICK(1);  // Z1bar MMA
      float dov[32];
      {
        uint32_t r[32];
        tmem_ld32(tmem + lane_addr + TM_DZQ + q0, r);
        tc_wait_ld();
        float z[32], ex[2] = {0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          z[e] = __uint_as_float(r[e]) + b1n[q0 + e];
          ex[0] += z[e];
          ex[1] = fmaf(z[e], z[e], ex[1]);
        }
        pair_rowsum<2>(xq + xsel * 256, gw, j, act, ex);
        xsel ^= 1;
        const float mu = ex[0] * (1.f / 64.f);
        const float rstd = rsqrtf(fmaxf(ex[1] * (1.f / 64.f) - mu * mu, 0.f) + 1e-8f);
        ld_row16(dot, j, 4 * gw, dov);
        ld_row16(dot, j, 4 * gw + 2, dov + 16);
        float sq[2] = {0.f, 0.f};
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          z[e] = (z[e] - mu) * rstd;  // x_hat of the output LayerNorm
          const float dxh = dov[e] * lnw[q0 + e];
          sq[0] += dxh;
          sq[1] = fmaf(dxh, z[e], sq[1]);
          if (act) {
            dgq[e] = fmaf(dov[e], z[e], dgq[e]);
            dbq[e] += dov[e];
          }
        }
        pair_rowsum<2>(xq + xsel * 256, gw, j, act, sq);
        xsel ^= 1;
        const float sc = rstd * (1.f / 64.f);
#pragma unroll
        for (int e = 0; e < 32; ++e) z[e] = (fmaf(64.f, dov[e] * lnw[q0 + e], -sq[0]) - z[e] * sq[1]) * sc;  // dZ1bar
        TICK(2);  // output-LN backward
        if (i >= 2) {  // factor-tile slot: the K side must have folded step i-2 (same slot) into the state gradient
          mbar_wait(&bar_qfree[ds], ((i >> 1) - 1) & 1);
          if (tid == 128 && i + 1 < nst) load_q(i + 1);  // ... which also released the Q / dOut slot of step i-2
        }
        if (act) {
          st_tok4(dzq, j, 4 * gw, z);
          st_tok4(dzq, j, 4 * gw + 2, z + 16);
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) z[e] = 0.f;
        }
        warp_colsum16(z, lane);
        warp_colsum16(z + 16, lane);
        if ((lane & 1) == 0) {
          qdb1[(i & 3) * 64 + q0 + (lane >> 1)] = z[0];
          qdb1[(i & 3) * 64 + q0 + 16 + (lane >> 1)] = z[16];
        }
      }
      fence_proxy_async();
      tc_fence_before();
      pair_sync();
      TICK(3);  // wait for the slot + tile write
      if (tid == 128) {
        mbar_arrive(&bar_qready[ds]);
        tc_fence_after();
        mma_kn(tmem + TM_DQ, dzq, img_n, false);  // d XQ = dZ1bar . W1'^T (+ dOut below)
        tc_commit(bar_mq);
      }
      mbar_wait(bar_mq, mq_phase);
      mq_phase ^= 1;
      tc_fence_after();
      TICK(4);  // dQ MMA
      {
        uint32_t r[32];
        tmem_ld32(tmem + lane_addr + TM_DQ + q0, r);
        tc_wait_ld();
        if (act) {
          float o[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) o[e] = __uint_as_float(r[e]) + dov[e];
          __nv_bfloat16* dst = p.dXQ + (((size_t)bh * NC + t) * CS + j) * F + q0;
          st_global16(dst, o);
          st_global16(dst + 16, o + 16);
        }
      }
      tc_fence_before();
      pair_sync();
      TICK(5);  // d XQ store
    }
    if (!act) {
#pragma unroll
      for (int e = 0; e < 32; ++e) { dgq[e] = 0.f; dbq[e] = 0.f; }
    }
    warp_colsum16(dgq, lane);
    warp_colsum16(dgq + 16, lane);
    warp_colsum16(dbq, lane);
    warp_colsum16(dbq + 16, lane);
    if ((lane & 1) == 0) {
      atomicAdd(p.dlnw + (size_t)bh * F + q0 + (lane >> 1), dgq[0]);
      atomicAdd(p.dlnw + (size_t)bh * F + q0 + 16 + (lane >> 1), dgq[16]);
      atomicAdd(p.dlnb + (size_t)bh * F + q0 + (lane >> 1), dbq[0]);
      atomicAdd(p.dlnb + (size_t)bh * F + q0 + 16 + (lane >> 1), dbq[16]);
    }
  }

  else if (elect_one()) {  // one lane of warp 6 (the branch above is warp-uniform)
    // =============================================== issue warp =====================================================
    for (int m = 0; m < 4; ++m)
      if (p.t_hi + 1 - m >= p.t_lo) load_image(p.t_hi + 1 - m);
    for (int i = 0; i < 3 && i < nst; ++i) load_k(i);
    const uint32_t gt = sbase + SM_G, dzt = sbase + SM_DZ, dwi = sbase + SM_DWI;
    mbar_wait(bar_kb, 0);  // state gradient loaded into TMEM
    tc_fence_after();
    mbar_wait(&bar_qready[0], 0);  // fold the Q side of the first step, then release the chain
    mma_upd(tmem + TM_DW, sbase + SM_DZQ, sbase + SM_QT);
    tc_commit(bar_upd);
    tc_commit(&bar_qfree[0]);
    mbar_wait(&bar_k[0], 0);
    mbar_wait(&bar_img[p.t_hi & 3], 0);
    mma_kk(tmem + TM_DZ, sbase + SM_KT, sbase + SM_IMG + (p.t_hi & 3) * 8192);
    tc_commit(bar_mz);
    for (int i = 0; i < nst; ++i) {
      const int t = p.t_hi - i;
      const uint32_t kt = sbase + SM_KT + (i % 3) * 16384;
      const uint32_t dk = tmem + ((i & 1) ? TM_DK1 : TM_DK0);
      // (C) dG = K . dW1' ; dK = G . dW1'^T ; then the next step's Z1 recompute
      mbar_wait(bar_kb, (i + 1) & 1);
      tc_fence_after();
      mma_kk(tmem + TM_DG, kt, dwi);
      mma_kn(dk, gt, dwi, false);
      tc_commit(bar_mg);
      if (i + 1 < nst) {
        mbar_wait(&bar_k[(i + 1) % 3], ((i + 1) / 3) & 1);
        mbar_wait(&bar_img[(t - 1) & 3], ((i + 2) >> 2) & 1);
        mma_kk(tmem + TM_DZ, sbase + SM_KT + ((i + 1) % 3) * 16384, sbase + SM_IMG + ((t - 1) & 3) * 8192);
        tc_commit(bar_mz);
      }
      if (i > 0) {  // the previous step's update is complete: refill the K / V slot and the image slot it released
        mbar_wait(bar_mkb, (i - 1) & 1);
        if (i + 2 < nst) load_k(i + 2);
        if (t - 2 >= p.t_lo) load_image(t - 2);
      }
      // (F) dK += dZ1 . W1^T ; dW^T += dZ1^T . K ; then fold the next step's Q-side factor
      mbar_wait(bar_ke, i & 1);
      tc_fence_after();
      mma_kn(dk, dzt, sbase + SM_IMG + (t & 3) * 8192, true);
      mma_upd(tmem + TM_DW, dzt, kt);
      tc_commit(bar_mkb);
      if (i + 1 < nst) {
        mbar_wait(&bar_qready[(i + 1) & 1], ((i + 1) >> 1) & 1);
        mma_upd(tmem + TM_DW, sbase + SM_DZQ + ((i + 1) & 1) * 16384, sbase + SM_QT + ((i + 1) % 3) * 16384);
        tc_commit(bar_upd);
        tc_commit(&bar_qfree[(i + 1) & 1]);
      }
    }
  }

  TICK_DUMP(12, p.dbg);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

}  // namespace linb

size_t linear_backward_window(int NC, int G) {  // steps per recompute window: a multiple of the checkpoint group
  if (G >= NC) return (size_t)NC;
  const int target = 256;
  return (size_t)(G >= target ? G : G * (target / G));
}

// window buffers: two (recompute of window w - 1 overlaps the reverse pass over window w) unless one window covers NC
static int linear_backward_buffers(int NC, int G) { return (size_t)NC > linear_backward_window(NC, G) ? kLinMaxBuffers : 1; }

size_t linear_backward_workspace_bytes(int B, int H, int NC, int G) {
  return carve_linear_workspace(nullptr, ((size_t)B * H + 1) / 2, linear_backward_window(NC, G) + 1,
                                linear_backward_buffers(NC, G), nullptr);
}

cudaError_t launch_linear_backward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                   const float* ln_b, const float* W1c, const float* b1c, const void* dOut, float* dlnw,
                                   float* dlnb, float* dW1, float* db1, float* dEta, void* dXQ, void* dXK, void* dXV,
                                   void* workspace, size_t workspace_bytes, int B, int H, int NC, int G,
                                   cudaStream_t stream) {
  if (B <= 0 || H <= 0 || NC <= 0 || G <= 0) { g_where = "bad sizes"; return cudaErrorInvalidValue; }
  if (G > NC) G = NC;
  const int BH = B * H;
  const uint64_t rows = (uint64_t)BH * NC * linb::CS;
  if (rows > 0x7FFFFFFFull) { g_where = "too many rows"; return cudaErrorInvalidValue; }
  if (workspace_bytes < linear_backward_workspace_bytes(B, H, NC, G)) { g_where = "workspace too small"; return cudaErrorInvalidValue; }
  CUtensorMap tq, tk, tv, tdo;
  if (make_token_tmap_box(&tq, XQ, rows, 16) || make_token_tmap_box(&tk, XK, rows, 16) || make_token_tmap_box(&tv, XV, rows, 16) ||
      make_token_tmap_box(&tdo, dOut, rows, 16))
    return cudaErrorInvalidValue;

  const int S = (int)linear_backward_window(NC, G);
  const int nwin = (NC + S - 1) / S;
  const int K = (NC + G - 1) / G;  // checkpoints per sequence
  const size_t slots = (size_t)S + 1;
  const int nbuf = linear_backward_buffers(NC, G);
  LinearImages img[kLinMaxBuffers];
  carve_linear_workspace(workspace, ((size_t)BH + 1) / 2, slots, nbuf, img);

  std::lock_guard<std::mutex> enqueue_lock(device_enqueue_mutex());
  static bool attr_done_dev[64] = {};  // function attributes (and side streams) are per device
  bool& attr_done = *device_once(attr_done_dev);
  struct Side { cudaStream_t sT; cudaEvent_t evT[2], evR[2], evIn; };
  static Side sides[64];
  int dev_ = 0;
  TB_TRY(cudaGetDevice(&dev_), "cudaGetDevice");
  Side& sd_ = sides[dev_ & 63];
  cudaStream_t& sT = sd_.sT;
  cudaEvent_t(&evT)[2] = sd_.evT;
  cudaEvent_t(&evR)[2] = sd_.evR;
  cudaEvent_t& evIn = sd_.evIn;
  if (!attr_done) {
    TB_TRY(cudaFuncSetAttribute(linb::ttt_linear_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, linb::SM_TOTAL), "smem attr");
    TB_TRY(cudaStreamCreateWithFlags(&sT, cudaStreamNonBlocking), "stream create");
    for (int b = 0; b < 2; ++b) {
      TB_TRY(cudaEventCreateWithFlags(&evT[b], cudaEventDisableTiming), "event create");
      TB_TRY(cudaEventCreateWithFlags(&evR[b], cudaEventDisableTiming), "event create");
    }
    TB_TRY(cudaEventCreateWithFlags(&evIn, cudaEventDisableTiming), "event create");
    attr_done = true;
  }
  // d ln_weight / d ln_bias are per-(batch, head) partials [B,H,64] accumulated with atomics; the caller sums over B
  TB_TRY(cudaMemsetAsync(dlnw, 0, (size_t)BH * 64 * sizeof(float), stream), "memset dlnw");
  TB_TRY(cudaMemsetAsync(dlnb, 0, (size_t)BH * 64 * sizeof(float), stream), "memset dlnb");
  TB_TRY(cudaEventRecord(evIn, stream), "event record");
  TB_TRY(cudaStreamWaitEvent(sT, evIn, 0), "stream wait");

  // trajectory of window w on the side stream (buffer w & 1), one window ahead of the reverse kernel
  auto recompute = [&](int w) -> cudaError_t {
    const int b = w % nbuf, t0 = w * S, n = (t0 + S <= NC ? S : NC - t0);
    if (w + nbuf < nwin) TB_TRY(cudaStreamWaitEvent(sT, evR[b], 0), "stream wait");  // buffer still read by window w + 2
    const int ck = t0 / G;
    cudaError_t e = launch_linear_trajectory(XK, XV, last_eta, ln_w, ln_b, W1c + (size_t)ck * 64 * 64, b1c + (size_t)ck * 64,
                                             (long long)K * 64 * 64, (long long)K * 64, img[b], (int)slots, B, H, NC,
                                             t0, n, sT);
    if (e != cudaSuccess) return e;
    TB_TRY(cudaEventRecord(evT[b], sT), "event record");
    return cudaSuccess;
  };
  cudaError_t e = recompute(nwin - 1);
  if (e != cudaSuccess) return e;
  for (int w = nwin - 1; w >= 0; --w) {
    const int b = w % nbuf, t0 = w * S, n = (t0 + S <= NC ? S : NC - t0);
    if (w > 0) { e = recompute(w - 1); if (e != cudaSuccess) return e; }
    TB_TRY(cudaStreamWaitEvent(stream, evT[b], 0), "stream wait");
    linb::LinBwdParams p{};
    p.last_eta = reinterpret_cast<const __nv_bfloat16*>(last_eta);
    p.ln_w = ln_w; p.ln_b = ln_b; p.in = img[b];
    p.dW1 = dW1; p.db1 = db1;
    p.dXQ = reinterpret_cast<__nv_bfloat16*>(dXQ); p.dXK = reinterpret_cast<__nv_bfloat16*>(dXK);
    p.dXV = reinterpret_cast<__nv_bfloat16*>(dXV); p.dEta = dEta; p.dlnw = dlnw; p.dlnb = dlnb;
    p.H = H; p.NC = NC; p.img_slots = (int)slots; p.t_hi = t0 + n - 1; p.t_lo = t0; p.t0 = t0; p.first = (w == nwin - 1);
    p.dbg = g_timing_buf;
    g_where = "linear backward launch";
    linb::ttt_linear_bwd_kernel<<<BH, linb::NT, linb::SM_TOTAL, stream>>>(tq, tk, tv, tdo, p);
    TB_TRY(cudaGetLastError(), "linear backward launch");
    TB_TRY(cudaEventRecord(evR[b], stream), "event record");
  }
  return cudaSuccess;
}

}  // namespace tb
