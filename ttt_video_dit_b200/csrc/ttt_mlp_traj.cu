// TTT-MLP trajectory recompute for the backward pass (sm_100a): replays the K side of the steps of one checkpoint group
// from the checkpointed fp32 state and saves the bf16 operand image of the state entering every step (what
// ttt-tk/kernels/ttt_backward/ttt.cu:1-260 re-materialises per group from its W checkpoints).  Same arithmetic and tile
// conventions as ttt_mlp_fwd.cu (K side only), but written for CODE SIZE, not speed:
//
// The backward pass runs three kernels concurrently (this one, the parallel Q-side kernel and the sequential K-side
// kernel).  Measured on B200 (profiles/r01_icache_interference_*.log): a co-running kernel whose loop body exceeds the
// SM's 32 KB L1.5 instruction cache streams its code through the chip-wide instruction path and slows the K-side kernel
// (whose own loop is 112 KB) by 45 %, even from a single SM; a loop of <= 28 KB has no measurable effect.  The unrolled
// forward kernel in trajectory mode has a 48 KB loop.  Here every per-thread element loop is a rolled loop over
// 16-column chunks (values that the forward keeps in registers across phases live in shared memory instead), which
// keeps the whole step loop inside L1.5.  This kernel has 2x slack against the K-side kernel, so the lost ILP is free.
//
// Operand format: as in the forward (template kF16, see ttt_mlp_fwd.cu) the MMA operand tiles of THIS kernel are fp16, so
// that the recomputed trajectory follows the forward's; the state images it exports for the K-side / Q-side kernels are
// bf16 (those kernels mix them with gradient operands, which need bf16's range), written by the owning threads straight
// to global memory in the image's tile byte order.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "bwd_common.cuh"
#include "ptx.cuh"
#include "recompute_ring.cuh"
#include "ttt_internal.h"

namespace tb {
namespace traj {

using bwd::gelu1;
using bwd::ld_row16;
using bwd::st_row16;
using bwd::warp_colsum16;

// operand-format variants of bwd_common.cuh's row helpers
template <bool kF16>
__device__ __forceinline__ void ld_row16_op(uint32_t tile, int row, int chunk0, float* v) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    uint32_t a, b, cc, d;
    ld_shared_v4(tile + sw128_off(row, chunk0 + c), a, b, cc, d);
    v[8 * c + 0] = op_lo<kF16>(a); v[8 * c + 1] = op_hi<kF16>(a); v[8 * c + 2] = op_lo<kF16>(b); v[8 * c + 3] = op_hi<kF16>(b);
    v[8 * c + 4] = op_lo<kF16>(cc); v[8 * c + 5] = op_hi<kF16>(cc); v[8 * c + 6] = op_lo<kF16>(d); v[8 * c + 7] = op_hi<kF16>(d);
  }
}
template <bool kF16>
__device__ __forceinline__ void st_row16_op(uint32_t tile, int row, int chunk0, const float* v) {
#pragma unroll
  for (int c = 0; c < 2; ++c)
    st_shared_v4(tile + sw128_off(row, chunk0 + c), pack_op<kF16>(v[8 * c], v[8 * c + 1]), pack_op<kF16>(v[8 * c + 2], v[8 * c + 3]),
                 pack_op<kF16>(v[8 * c + 4], v[8 * c + 5]), pack_op<kF16>(v[8 * c + 6], v[8 * c + 7]));
}
// 16 fp32 of row `row` -> bf16 -> the two 16-byte chunks chunk0, chunk0+1 of a [256][64] image block in global memory
__device__ __forceinline__ void st_image16(uint8_t* img_block, int row, int chunk0, const float* v) {
#pragma unroll
  for (int c = 0; c < 2; ++c)
    *reinterpret_cast<uint4*>(img_block + sw128_off(row, chunk0 + c)) =
        make_uint4(pack_bf16(v[8 * c], v[8 * c + 1]), pack_bf16(v[8 * c + 2], v[8 * c + 3]), pack_bf16(v[8 * c + 4], v[8 * c + 5]),
                   pack_bf16(v[8 * c + 6], v[8 * c + 7]));
}
__device__ __forceinline__ void tile_bf16_to_f16(uint32_t tile_saddr, int tid) {  // [64][64] tile, in place
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const uint32_t a = tile_saddr + (uint32_t)(tid + 256 * i) * 16u;
    uint32_t w0, w1, w2, w3;
    ld_shared_v4(a, w0, w1, w2, w3);
    st_shared_v4(a, bf16x2_to_f16x2(w0), bf16x2_to_f16x2(w1), bf16x2_to_f16x2(w2), bf16x2_to_f16x2(w3));
  }
}

constexpr int CS = 64, F = 64, HID = 256, NT = 256;

constexpr uint32_t SM_W1B = 0;                 // W1^T bf16 [256][64]  (image block 0)
constexpr uint32_t SM_W2B = 32768;             // W2   bf16 [256][64]  (image block 1)
constexpr uint32_t SM_X2 = 65536;              // X2^T [256 hidden][64 tok]
constexpr uint32_t SM_GP = SM_X2 + 32768;      // gelu'(Z1)^T, overwritten in place by G1^T
constexpr uint32_t SM_K = SM_GP + 32768;       // 2 slots x K_t [64][64]
constexpr uint32_t SM_V = SM_K + 2 * 8192;     // 2 slots x V_t [64][64]
constexpr uint32_t SM_G2 = SM_V + 2 * 8192;    // G2 = -eta * gradZ2 [64 tok][64]
constexpr uint32_t SM_MISC = SM_G2 + 8192;     // b2[64], ln_w[64], ln_b[64], db2acc[64], barriers, tmem ptr
constexpr uint32_t SM_XB = SM_MISC + 2048;     // LN exchange: float2[2][64] x 2
constexpr uint32_t SM_TOTAL = SM_XB + 2048;

constexpr uint32_t TM_W1 = 0, TM_W2 = 128, TM_D1 = 256, TM_D3 = 256, TM_D2 = 384;  // D1/D3: + 64 * half

struct TrajParams {
  const __nv_bfloat16* last_eta;        // [B,H,NC,64]
  const float *ln_w, *ln_b;             // [H,64]
  const float *W1, *b1, *W2, *b2;       // checkpoint arrays [BH][K]...
  int NC, H, K, G, t0, t_end, img_slots;  // one checkpoint group: steps [t0, t_end), t0 = checkpoint index * G
  MlpSlot slot;                         // receives the images of the states entering steps t0 .. t_end (recompute_ring.cuh)
  // persistent K-side mode: [BH] flags of the unit that used this ring slot before; the CTA of sequence bh starts writing
  // only after the K-side CTA of bh has released the slot (null: the host orders the launches with events instead)
  const unsigned* wait_done;
};

template <bool kF16>
__global__ void __launch_bounds__(NT, 1)
ttt_mlp_traj_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV, const TrajParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = uniform_warp_id();  // == warp, provably warp-uniform: single-thread issue blocks branch on it
  const int bh = blockIdx.x, head = bh % p.H;
  const int n = p.t_end - p.t0;
  const int half = warp >> 2, j = tid;
  const uint32_t lane_addr = ((uint32_t)((warp & 3) * 32)) << 16;

  if (p.wait_done != nullptr) {
    if (tid == 0) wait_flag<512>(p.wait_done + bh, 1);
    __syncthreads();
  }
  float* b2s = reinterpret_cast<float*>(smem + SM_MISC);
  float* lnw = b2s + 64;
  float* lnb = lnw + 64;
  float* db2acc = lnb + 64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_MISC + 1024);
  uint64_t* tma_bar = bars;      // [2]
  uint64_t* mma_bar = bars + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 4);
  float2* xs1 = reinterpret_cast<float2*>(smem + SM_XB);         // [2][64] (sum z, sum z^2) per column half
  float2* xs2 = reinterpret_cast<float2*>(smem + SM_XB + 1024);  // [2][64] (s1, s2)

  if (warp_u == 0 && elect_one()) {
    mbar_init(&tma_bar[0], 1);
    mbar_init(&tma_bar[1], 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 0) tmem_alloc<512>(tmem_ptr);
  const size_t st = (size_t)bh * p.K + (size_t)(p.t0 / p.G);
  if (tid < 64) {
    lnw[tid] = p.ln_w[head * 64 + tid];
    lnb[tid] = p.ln_b[head * 64 + tid];
    b2s[tid] = p.b2[st * 64 + tid];
    db2acc[tid] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  const size_t row_base = ((size_t)bh * p.NC + p.t0) * CS;
  uint8_t* img = p.slot.image(bh, p.img_slots, 0);
  float* b1img = p.slot.image_b1(bh, p.img_slots, 0);
  float* b2img = p.slot.image_b2(bh, p.img_slots, 0);

  if (warp_u == 0 && elect_one()) {
    mbar_expect_tx(&tma_bar[0], 16384);
    tma_load_2d(smem + SM_K, &tmK, 0, (int)row_base, &tma_bar[0]);
    tma_load_2d(smem + SM_V, &tmV, 0, (int)row_base, &tma_bar[0]);
  }

  // ---- checkpointed state -> TMEM accumulators + bf16 operand copies (= image record 0)
  float b1r = p.b1[st * HID + j];
  {
    const float* W1g = p.W1 + st * F * HID;
    const float* W2g = p.W2 + st * HID * F;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      float v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = W1g[(size_t)(16 * c + i) * HID + j];
      tmem_st16(tmem + lane_addr + TM_W1 + 64 * half + 16 * c, reinterpret_cast<uint32_t*>(v));
      st_row16_op<kF16>(sbase + SM_W1B, j, 2 * c, v);
      st_image16(img + kImageW1T, j, 2 * c, v);  // image of the state entering step t0
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = W2g[(size_t)j * F + 16 * c + i];
      tmem_st16(tmem + lane_addr + TM_W2 + 64 * half + 16 * c, reinterpret_cast<uint32_t*>(v));
      st_row16_op<kF16>(sbase + SM_W2B, j, 2 * c, v);
      st_image16(img + kImageW2, j, 2 * c, v);
    }
    b1img[j] = b1r;
    if (tid < 64) b2img[tid] = b2s[tid];
    tc_wait_st();
  }
  if (kF16) {  // K_0 landed during the state staging: bf16 -> f16 in place (V is not an MMA operand and stays bf16)
    mbar_wait(&tma_bar[0], 0);
    tile_bf16_to_f16(sbase + SM_K, tid);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();

  constexpr uint32_t IDESC_KK = make_idesc_bf16(128, 64, false, false, false, kF16, kF16);  // A K-major, B K-major
  constexpr uint32_t IDESC_NN = make_idesc_bf16(128, 64, true, true, false, kF16, kF16);    // A MN-major, B MN-major
  constexpr uint32_t IDESC_KN = make_idesc_bf16(128, 64, false, true, false, kF16, kF16);   // A K-major, B MN-major
  uint32_t mma_phase = 0;

  // D1[h] = W1b^T[h] . K^T  (M = 128 hidden, N = 64 tokens, K = 64)
  auto issue_p1 = [&](int it_next) {
    const int sl = it_next & 1;
    mbar_wait(&tma_bar[sl], (it_next >> 1) & 1);
    tc_fence_after();
    const uint64_t db = make_desc_sw128(sbase + SM_K + sl * 8192, 16, 1024);
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      const uint64_t da = make_desc_sw128(sbase + SM_W1B + h * 16384, 16, 1024);
#pragma unroll 1
      for (int k = 0; k < 4; ++k) umma_ss(tmem + TM_D1 + 64 * h, desc_advance(da, 32 * k), desc_advance(db, 32 * k), IDESC_KK, k > 0);
    }
    tc_commit(mma_bar);
  };
  if (warp_u == 0 && elect_one()) issue_p1(0);

#pragma unroll 1
  for (int it = 0; it < n; ++it) {
    const int slot = it & 1;
    const uint32_t kt = sbase + SM_K + slot * 8192, vt = sbase + SM_V + slot * 8192;
    // LN threads: token row r (K side only: rows 0-63 -> warps 0,1 and 4,5), column half ch
    const int r = 32 * (warp & 3) + lane, ch = warp >> 2;
    const bool ln_thread = (warp & 3) < 2;
    unsigned short eta_raw = 0;
    if (ln_thread) eta_raw = reinterpret_cast<const unsigned short*>(p.last_eta)[row_base + (size_t)it * CS + r];

    mbar_wait(&tma_bar[slot], (it >> 1) & 1);
    if (warp_u == 0 && (it + 1 < n) && elect_one()) {
      const int ns = slot ^ 1;
      mbar_expect_tx(&tma_bar[ns], 16384);
      tma_load_2d(smem + SM_K + ns * 8192, &tmK, 0, (int)(row_base + (size_t)(it + 1) * CS), &tma_bar[ns]);
      tma_load_2d(smem + SM_V + ns * 8192, &tmV, 0, (int)(row_base + (size_t)(it + 1) * CS), &tma_bar[ns]);
    }
    mbar_wait(mma_bar, mma_phase);  // P1 (issued in the prologue / at the end of the previous step)
    mma_phase ^= 1;
    tc_fence_after();

    // ---- P2: X2^T = gelu(Z1^T) (bf16 tile), gelu'(Z1)^T (bf16, SM_GP)
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      float v[16], g[16];
      tmem_ld16(tmem + lane_addr + TM_D1 + 64 * half + 16 * c, reinterpret_cast<uint32_t*>(v));
      tc_wait_ld();
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = gelu1(v[i] + b1r, g[i]);
      st_row16_op<kF16>(sbase + SM_X2, j, 2 * c, v);
      st_row16(sbase + SM_GP, j, 2 * c, g);  // gelu' is not an operand (bf16); overwritten by G1^T in P6
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();

    // ---- P3: D2 = X2 . W2b  (M = 128: rows 64-127 come from the SM_GP block and are ignored; N = 64; K = 256)
    if (warp_u == 0 && elect_one()) {
      tc_fence_after();
      const uint64_t da = make_desc_sw128(sbase + SM_X2, 32768, 1024);
      const uint64_t db = make_desc_sw128(sbase + SM_W2B, 1024, 1024);
#pragma unroll 1
      for (int k = 0; k < 16; ++k) umma_ss(tmem + TM_D2, desc_advance(da, 2048 * k), desc_advance(db, 2048 * k), IDESC_NN, k > 0);
      tc_commit(mma_bar);
    }
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();

    // ---- P4: LayerNorm + L2 gradient on token rows (three rolled passes over the thread's 32 columns; Z2 is re-read
    //          from TMEM instead of being held in registers)
    float mu = 0.f, rstd = 0.f, s1 = 0.f, s2 = 0.f;
    if (ln_thread) {
      float a1 = 0.f, a2 = 0.f;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        float z[16];
        tmem_ld16(tmem + lane_addr + TM_D2 + 32 * ch + 16 * c, reinterpret_cast<uint32_t*>(z));
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) { z[i] += b2s[32 * ch + 16 * c + i]; a1 += z[i]; a2 = fmaf(z[i], z[i], a2); }
      }
      xs1[ch * 64 + r] = make_float2(a1, a2);
    }
    __syncthreads();
    if (ln_thread) {
      const float2 p0 = xs1[r], p1 = xs1[64 + r];
      mu = (p0.x + p1.x) * (1.0f / 64.0f);
      rstd = rsqrtf(fmaxf((p0.y + p1.y) * (1.0f / 64.0f) - mu * mu, 0.f) + 1e-8f);
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        float z[16], kk[16], vv[16];
        tmem_ld16(tmem + lane_addr + TM_D2 + 32 * ch + 16 * c, reinterpret_cast<uint32_t*>(z));
        ld_row16_op<kF16>(kt, r, 4 * ch + 2 * c, kk);
        ld_row16(vt, r, 4 * ch + 2 * c, vv);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int f = 32 * ch + 16 * c + i;
          const float xh = (z[i] + b2s[f] - mu) * rstd;
          const float g = (fmaf(lnw[f], xh, lnb[f]) - (vv[i] - kk[i])) * lnw[f];
          s1 += g;
          s2 = fmaf(g, xh, s2);
        }
      }
      xs2[ch * 64 + r] = make_float2(s1, s2);
    }
    __syncthreads();
    if (ln_thread) {
      const float2 p0 = xs2[r], p1 = xs2[64 + r];
      s1 = p0.x + p1.x; s2 = p0.y + p1.y;
      const float sc = -__uint_as_float((uint32_t)eta_raw << 16) * rstd * (1.0f / 64.0f);
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        float z[16], kk[16], vv[16];
        tmem_ld16(tmem + lane_addr + TM_D2 + 32 * ch + 16 * c, reinterpret_cast<uint32_t*>(z));
        ld_row16_op<kF16>(kt, r, 4 * ch + 2 * c, kk);
        ld_row16(vt, r, 4 * ch + 2 * c, vv);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int f = 32 * ch + 16 * c + i;
          const float xh = (z[i] + b2s[f] - mu) * rstd;
          const float g = (fmaf(lnw[f], xh, lnb[f]) - (vv[i] - kk[i])) * lnw[f];
          z[i] = (fmaf(64.0f, g, -s1) - xh * s2) * sc;  // G2 = -eta * gradZ2
        }
        st_row16_op<kF16>(sbase + SM_G2, r, 4 * ch + 2 * c, z);
        warp_colsum16(z, lane);  // b2 update = column sums of G2 over the token rows
        if ((lane & 1) == 0) atomicAdd(&db2acc[32 * ch + 16 * c + (lane >> 1)], z[0]);
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();

    // ---- P5: D3[h] = W2b[h] . G2^T ;  W2[h] += X2^T[h] . G2
    if (warp_u == 0 && elect_one()) {
      tc_fence_after();
      const uint64_t dg_k = make_desc_sw128(sbase + SM_G2, 16, 1024);
      const uint64_t dg_mn = make_desc_sw128(sbase + SM_G2, 1024, 1024);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const uint64_t da = make_desc_sw128(sbase + SM_W2B + h * 16384, 16, 1024);
#pragma unroll 1
        for (int k = 0; k < 4; ++k) umma_ss(tmem + TM_D3 + 64 * h, desc_advance(da, 32 * k), desc_advance(dg_k, 32 * k), IDESC_KK, k > 0);
      }
      tc_commit(mma_bar);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const uint64_t da = make_desc_sw128(sbase + SM_X2 + h * 16384, 16, 1024);
#pragma unroll 1
        for (int k = 0; k < 4; ++k) umma_ss(tmem + TM_W2 + 64 * h, desc_advance(da, 32 * k), desc_advance(dg_mn, 2048 * k), IDESC_KN, 1);
      }
    }
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();

    // ---- P6: G1^T = D3 * gelu'(Z1)^T in place over SM_GP ; b1 += row sum ; b2 += column sums of G2
    {
      float acc = 0.f;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        float v[16], g[16];
        tmem_ld16(tmem + lane_addr + TM_D3 + 64 * half + 16 * c, reinterpret_cast<uint32_t*>(v));
        ld_row16(sbase + SM_GP, j, 2 * c, g);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) { v[i] *= g[i]; acc += v[i]; }
        st_row16_op<kF16>(sbase + SM_GP, j, 2 * c, v);
      }
      b1r += acc;
      if (tid < 64) {
        b2s[tid] += db2acc[tid];
        db2acc[tid] = 0.f;
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();

    // ---- P7: W1^T[h] += G1^T[h] . K
    if (warp_u == 0 && elect_one()) {
      tc_fence_after();
      const uint64_t db = make_desc_sw128(kt, 1024, 1024);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const uint64_t da = make_desc_sw128(sbase + SM_GP + h * 16384, 16, 1024);
#pragma unroll 1
        for (int k = 0; k < 4; ++k) umma_ss(tmem + TM_W1 + 64 * h, desc_advance(da, 32 * k), desc_advance(db, 2048 * k), IDESC_KN, 1);
      }
      tc_commit(mma_bar);  // also covers the W2 update issued in P5
    }
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();

    // ---- P8: operand copies of the new state (smem) + its bf16 image (global) = image record it + 1 (the last one is
    //          the next group's checkpoint, read by the Q-side kernel of step t_end - 1)
    uint8_t* img_n = img + (size_t)(it + 1) * kImageBytes;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      float v[16];
      tmem_ld16(tmem + lane_addr + TM_W1 + 64 * half + 16 * c, reinterpret_cast<uint32_t*>(v));
      tc_wait_ld();
      st_row16_op<kF16>(sbase + SM_W1B, j, 2 * c, v);
      st_image16(img_n + kImageW1T, j, 2 * c, v);
    }
    if (kF16 && it + 1 < n) {  // next step's K tile (TMA issued at the top of this step): bf16 -> f16 in place
      mbar_wait(&tma_bar[slot ^ 1], ((it + 1) >> 1) & 1);
      tile_bf16_to_f16(sbase + SM_K + (slot ^ 1) * 8192, tid);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp_u == 0 && (it + 1 < n) && elect_one()) issue_p1(it + 1);  // runs under the W2 conversion below
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      float v[16];
      tmem_ld16(tmem + lane_addr + TM_W2 + 64 * half + 16 * c, reinterpret_cast<uint32_t*>(v));
      tc_wait_ld();
      st_row16_op<kF16>(sbase + SM_W2B, j, 2 * c, v);
      st_image16(img_n + kImageW2, j, 2 * c, v);
    }
    b1img[(size_t)(it + 1) * kImageB1Floats + j] = b1r;
    if (tid < 64) b2img[(size_t)(it + 1) * kImageB2Floats + tid] = b2s[tid];  // b2s was updated by the same thread in P6
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

}  // namespace traj

cudaError_t launch_mlp_trajectory_compact(const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                          const float* ln_b, const float* W1c, const float* b1c, const float* W2c,
                                          const float* b2c, int B, int H, int NC, int K, int G, int t0, int t_end,
                                          const MlpSlot& slot, cudaStream_t stream, const unsigned* wait_done) {
  if (G <= 0 || t0 < 0 || t0 >= NC || t0 % G != 0 || t_end != group_end(t0 / G, G, NC)) {
    g_where = "trajectory window is not one checkpoint group";
    return cudaErrorInvalidValue;
  }
  const uint64_t rows = (uint64_t)B * H * NC * traj::CS;
  CUtensorMap tk, tv;
  if (make_token_tmap(&tk, XK, rows) || make_token_tmap(&tv, XV, rows)) return cudaErrorInvalidValue;
  traj::TrajParams p{};
  p.last_eta = reinterpret_cast<const __nv_bfloat16*>(last_eta);
  p.ln_w = ln_w; p.ln_b = ln_b; p.W1 = W1c; p.b1 = b1c; p.W2 = W2c; p.b2 = b2c;
  p.NC = NC; p.H = H; p.K = K; p.G = G; p.t0 = t0; p.t_end = t_end; p.img_slots = G + 1;
  p.slot = slot; p.wait_done = wait_done;
  static bool attr_done_dev[64] = {};  // function attributes (and side streams) are per device
  bool& attr_done = *device_once(attr_done_dev);
  if (!attr_done) {
    TB_TRY(cudaFuncSetAttribute(traj::ttt_mlp_traj_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, traj::SM_TOTAL), "smem attr (traj)");
    TB_TRY(cudaFuncSetAttribute(traj::ttt_mlp_traj_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, traj::SM_TOTAL), "smem attr (traj)");
    attr_done = true;
  }
  g_where = "trajectory launch";
  if (mlp_operands_bf16()) traj::ttt_mlp_traj_kernel<false><<<B * H, traj::NT, traj::SM_TOTAL, stream>>>(tk, tv, p);
  else                     traj::ttt_mlp_traj_kernel<true><<<B * H, traj::NT, traj::SM_TOTAL, stream>>>(tk, tv, p);
  return cudaGetLastError();
}

}  // namespace tb
