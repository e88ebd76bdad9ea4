// TTT-MLP backward, Q-side kernel (parallel over steps).
//
// The backward of the *output* half of step s (Zbar1 = Q W' + b', Xbar2 = gelu, Zbar2, LN, +Q residual; SURVEY appendix
// B stages 4 and 3a) depends only on the state AFTER step s (image W_{s+1}), on Q_s and on dOut_s -- not on the carried
// state gradient.  It is therefore taken off the sequential reverse chain: one CTA per (sequence, step) computes
//   dQ_s (final), the factor tiles Xbar2^T, dZbar2, dZbar1^T whose outer products the sequential kernel accumulates into
//   dW2 / dW1^T with two MMAs, the b1/b2 contributions, and the LN-parameter gradients of the output LayerNorm.
// grid = (steps of the group, B*H) fills the SMs the 48-CTA sequential kernels leave idle, and keeps the sequential
// kernel's code small enough for the instruction cache (measured: removing this code from the reverse kernel halves
// the time of its remaining phases, profiles/r01_phase_timing_bwd_noQ_experiment.log).
// Reference: the same math lives inside bwd_ttt_mlp_ker (ttt-tk/kernels/ttt_backward/ttt.cu:824-1100).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "bwd_common.cuh"
#include "ptx.cuh"
#include "recompute_ring.cuh"
#include "ttt_internal.h"

namespace tb {
namespace bwd {

constexpr uint32_t QS_W1I = 0;        // W1^T image of W_{s+1}     32 KB
constexpr uint32_t QS_W2I = 32768;    // W2 image                  32 KB
constexpr uint32_t QS_XB = 65536;     // Xbar2^T tile [256][64]    32 KB
constexpr uint32_t QS_ZB = 98304;     // dZbar1^T tile [256][64]   32 KB
constexpr uint32_t QS_TQ = 131072;    // Q_s [64][64]               8 KB
constexpr uint32_t QS_TDO = 139264;   // dOut_s                     8 KB
constexpr uint32_t QS_TT0 = 147456;   // dZbar2 [64][64]            8 KB
constexpr uint32_t QS_MISC = 155648;  // small vectors, exchange buffers, barriers (8 KB)
constexpr uint32_t QS_TOTAL = QS_MISC + 8192;
constexpr uint32_t QT_S0 = 0, QT_S1 = 64, QT_S2 = 128;  // TMEM working slots (256 columns allocated)

struct BwdQParams {
  const float *ln_w, *ln_b;      // [H,64]
  MlpSlot slot;                  // reads the state images, writes the factor records (recompute_ring.cuh)
  __nv_bfloat16* dXQ;            // out
  int H, NC, img_slots, G, t0;   // step s = t0 + blockIdx.x reads image record blockIdx.x + 1
  unsigned* ready;               // persistent K-side mode: counter [BH] of this unit, +1 per finished CTA (may be null)
};

// rolled (code-size) versions of bwd_common.cuh's mma_hid (N = 64, B K-major, no accumulate) and mma_tok
__device__ __forceinline__ void mma_hid_rolled(uint32_t d0, uint32_t d1, uint32_t a_tile, uint32_t b_tile) {
  constexpr uint32_t idesc = make_idesc_bf16(128, 64, false, false);
  const uint64_t db = make_desc_sw128(b_tile, 16, 1024);
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {
    const uint64_t da = make_desc_sw128(a_tile + h * 16384, 16, 1024);
#pragma unroll 1
    for (int k = 0; k < 4; ++k) umma_ss(h ? d1 : d0, desc_advance(da, 32 * k), desc_advance(db, 32 * k), idesc, k > 0);
  }
}
__device__ __forceinline__ void mma_tok_rolled(uint32_t d, uint32_t a_tile, uint32_t b_tile) {
  constexpr uint32_t idesc = make_idesc_bf16(128, 64, true, true);
  const uint64_t da = make_desc_sw128(a_tile, 0, 1024);
  const uint64_t db = make_desc_sw128(b_tile, 1024, 1024);
#pragma unroll 1
  for (int k = 0; k < 16; ++k) umma_ss(d, desc_advance(da, 2048 * k), desc_advance(db, 2048 * k), idesc, k > 0);
}

__global__ void __launch_bounds__(256, 1)
ttt_mlp_bwd_q_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO, const BwdQParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = uniform_warp_id();  // == warp, provably warp-uniform: single-thread issue blocks branch on it
  const int sl = blockIdx.x, bh = blockIdx.y, head = bh % p.H;
  const int s = p.t0 + sl;
  const int half = warp >> 2;
  const uint32_t lane_addr = ((uint32_t)((warp & 3) * 32)) << 16;
  const int j = tid;
  const int trow = 32 * (warp & 1) + lane, cq = 2 * (warp >> 2) + ((warp >> 1) & 1), c0 = 16 * cq;

  float* lnw = reinterpret_cast<float*>(smem + QS_MISC);
  float* lnb = lnw + 64;
  float* b2t = lnb + 64;
  float* cb2 = b2t + 64;   // column sums of dZbar2
  float* cgam = cb2 + 64;  // d gamma / d beta contributions of this step
  float* cbet = cgam + 64;
  float4* xA = reinterpret_cast<float4*>(smem + QS_MISC + 2048);  // [4][64]
  float2* xB = reinterpret_cast<float2*>(smem + QS_MISC + 6144);  // [4][64] (2 KB)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + QS_MISC + 1536);
  uint64_t* mma_bar = bars;
  uint64_t* bar_w = bars + 1;
  uint64_t* bar_qd = bars + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 4);

  if (warp_u == 0 && elect_one()) {
    mbar_init(mma_bar, 1);
    mbar_init(bar_w, 1);
    mbar_init(bar_qd, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmDO);
  }
  if (warp == 0) tmem_alloc<256>(tmem_ptr);
  const float* b2rec = p.slot.image_b2(bh, p.img_slots, sl + 1);
  const float* b1rec = p.slot.image_b1(bh, p.img_slots, sl + 1);
  if (tid < 64) {
    lnw[tid] = p.ln_w[head * 64 + tid];
    lnb[tid] = p.ln_b[head * 64 + tid];
    b2t[tid] = b2rec[tid];
    cb2[tid] = 0.f; cgam[tid] = 0.f; cbet[tid] = 0.f;
  }
  const float b1t = b1rec[j];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  const size_t row = ((size_t)bh * p.NC + s) * 64;
  if (warp_u == 0 && elect_one()) {
    const uint8_t* im = p.slot.image(bh, p.img_slots, sl + 1);
    mbar_expect_tx(bar_w, kImageBytes);
    bulk_load_1d(smem + QS_W1I, im + kImageW1T, 32768, bar_w);
    bulk_load_1d(smem + QS_W2I, im + kImageW2, 32768, bar_w);
    mbar_expect_tx(bar_qd, 16384);
    tma_load_2d(smem + QS_TQ, &tmQ, 0, (int)row, bar_qd);
    tma_load_2d(smem + QS_TDO, &tmDO, 0, (int)row, bar_qd);
  }
  uint32_t mma_phase = 0;
  mbar_wait(bar_w, 0);
  mbar_wait(bar_qd, 0);

  // ===== Q1 MMA: Zbar1^T = W1 . Q^T -> (S0,S1)
  if (warp_u == 0 && elect_one()) {
    tc_fence_after();
    mma_hid_rolled(tmem + QT_S0, tmem + QT_S1, sbase + QS_W1I, sbase + QS_TQ);
    tc_commit(mma_bar);
  }
  MMA_WAIT();
  // ===== Q2 [H]: Xbar2 tile, gelu'(Zbar1) (bf16, parked in the ZB tile until Q6 overwrites it in place).  Rolled
  //       16-column chunks: this kernel must stay inside the 32 KB L1.5 instruction cache (see ttt_mlp_traj.cu)
  {
    const uint32_t src = tmem + lane_addr + (half ? QT_S1 : QT_S0);
#pragma unroll 1
    for (int c = 0; c < 8; ++c) {  // one 16-byte chunk (8 tokens) per trip
      float v[8], g[8];
      tmem_ld8(src + 8 * c, reinterpret_cast<uint32_t*>(v));
      tc_wait_ld();
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = gelu1(v[i] + b1t, g[i]);
      st_shared_v4(sbase + QS_XB + sw128_off(j, c), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
      st_shared_v4(sbase + QS_ZB + sw128_off(j, c), pack_bf16(g[0], g[1]), pack_bf16(g[2], g[3]), pack_bf16(g[4], g[5]), pack_bf16(g[6], g[7]));
    }
  }
  PHASE_SYNC();
  // ===== Q3 MMA: Zbar2 = Xbar2 . W2 -> S2 (rows duplicated on lanes 64-127)
  if (warp_u == 0 && elect_one()) {
    tc_fence_after();
    mma_tok_rolled(tmem + QT_S2, sbase + QS_XB, sbase + QS_W2I);
    tc_commit(mma_bar);
  }
  MMA_WAIT();
  // ===== Q4 [T] (all warps): output LN backward: dZbar2 -> TT0 ; column sums for d b2, d gamma, d beta
  {
    float z[16], d[16];
    tmem_ld16(tmem + lane_addr + QT_S2 + c0, reinterpret_cast<uint32_t*>(z));
    ld_row16(sbase + QS_TDO, trow, 2 * cq, d);
    tc_wait_ld();
    float a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int f = 0; f < 16; ++f) { z[f] += b2t[c0 + f]; a1 += z[f]; a2 = fmaf(z[f], z[f], a2); }
    xB[cq * 64 + trow] = make_float2(a1, a2);
    __syncthreads();
    a1 = 0.f; a2 = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) { const float2 v = xB[q * 64 + trow]; a1 += v.x; a2 += v.y; }
    const float mu = a1 * (1.f / 64.f);
    const float rstd = rsqrtf(fmaxf(a2 * (1.f / 64.f) - mu * mu, 0.f) + 1e-8f);
    float s1 = 0.f, s2 = 0.f;
    float cg[16];
#pragma unroll
    for (int f = 0; f < 16; ++f) {
      z[f] = (z[f] - mu) * rstd;
      cg[f] = d[f] * z[f];
      const float dxh = d[f] * lnw[c0 + f];
      s1 += dxh;
      s2 = fmaf(dxh, z[f], s2);
    }
    xA[cq * 64 + trow] = make_float4(s1, s2, 0.f, 0.f);
    __syncthreads();
    s1 = 0.f; s2 = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) { const float4 v = xA[q * 64 + trow]; s1 += v.x; s2 += v.y; }
#pragma unroll
    for (int f = 0; f < 16; ++f) z[f] = (fmaf(64.f, d[f] * lnw[c0 + f], -s1) - z[f] * s2) * (rstd * (1.f / 64.f));  // dZbar2
    st_row16(sbase + QS_TT0, trow, 2 * cq, z);
    warp_colsum16(z, lane);
    warp_colsum16(cg, lane);
    warp_colsum16(d, lane);
    if ((lane & 1) == 0) {
      const int f = c0 + (lane >> 1);
      atomicAdd(&cb2[f], z[0]);
      atomicAdd(&cgam[f], cg[0]);
      atomicAdd(&cbet[f], d[0]);
    }
  }
  PHASE_SYNC();
  // ===== Q5 MMA: dXbar2^T = W2 . dZbar2^T -> (S0,S1)
  if (warp_u == 0 && elect_one()) {
    tc_fence_after();
    mma_hid_rolled(tmem + QT_S0, tmem + QT_S1, sbase + QS_W2I, sbase + QS_TT0);
    tc_commit(mma_bar);
  }
  MMA_WAIT();
  // ===== Q6 [H]: dZbar1 = dXbar2 * gelu'(Zbar1) -> ZB tile (in place) ; sum_i dZbar1 -> qb1
  {
    const uint32_t src = tmem + lane_addr + (half ? QT_S1 : QT_S0);
    float acc = 0.f;
#pragma unroll 1
    for (int c = 0; c < 8; ++c) {
      float v[8];
      uint32_t g0, g1, g2, g3;
      tmem_ld8(src + 8 * c, reinterpret_cast<uint32_t*>(v));
      ld_shared_v4(sbase + QS_ZB + sw128_off(j, c), g0, g1, g2, g3);
      tc_wait_ld();
      v[0] *= bf16_lo(g0); v[1] *= bf16_hi(g0); v[2] *= bf16_lo(g1); v[3] *= bf16_hi(g1);
      v[4] *= bf16_lo(g2); v[5] *= bf16_hi(g2); v[6] *= bf16_lo(g3); v[7] *= bf16_hi(g3);
      acc += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
      st_shared_v4(sbase + QS_ZB + sw128_off(j, c), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    }
    p.slot.factor_b1(bh, p.G, sl)[j] = acc;
  }
  PHASE_SYNC();
  // ===== Q7 MMA: dQ_u = dZbar1 . W1 -> S2 ; factor tiles -> global scratch
  if (warp_u == 0 && elect_one()) {
    tc_fence_after();
    mma_tok_rolled(tmem + QT_S2, sbase + QS_ZB, sbase + QS_W1I);
    tc_commit(mma_bar);
    uint8_t* dst = p.slot.factors(bh, p.G, sl);
    bulk_store_1d(dst + kFactorXbar2T, smem + QS_XB, 32768);
    bulk_store_1d(dst + kFactorDZbar1T, smem + QS_ZB, 32768);
    bulk_store_1d(dst + kFactorDZbar2, smem + QS_TT0, 8192);
    bulk_commit();
  }
  if (tid < 64) {
    // per-step partials, added by the sequential K-side kernel in step order (no global atomics: the LayerNorm parameter
    // gradients are bitwise reproducible); the shared-memory sums above start from zero and take exactly two addends
    float* q2 = p.slot.factor_vec(bh, p.G, sl);
    q2[kFactorDb2 + tid] = cb2[tid];
    q2[kFactorDgamma + tid] = cgam[tid];
    q2[kFactorDbeta + tid] = cbet[tid];
  }
  MMA_WAIT();
  // ===== Q8 [T]: dQ = dO + dQ_u
  {
    float a[16], d[16];
    tmem_ld16(tmem + lane_addr + QT_S2 + c0, reinterpret_cast<uint32_t*>(a));
    ld_row16(sbase + QS_TDO, trow, 2 * cq, d);
    tc_wait_ld();
#pragma unroll
    for (int f = 0; f < 16; ++f) a[f] += d[f];
    st_global16(p.dXQ + (row + trow) * 64 + c0, a);
  }
  // the factor tiles must have landed in global memory (not only been read out of smem) before this CTA is reported done
  if (warp_u == 0 && elect_one()) bulk_wait<0>();
  tc_fence_before();
  __syncthreads();
  if (p.ready != nullptr && tid == 0) release_flag<kCount>(p.ready + bh);  // every thread's global stores precede the barrier above
  if (warp == 0) tmem_dealloc<256>(tmem);
}

}  // namespace bwd

cudaError_t launch_mlp_backward_q(const CUtensorMap& tq, const CUtensorMap& tdo, const float* ln_w, const float* ln_b,
                                  const MlpSlot& slot, void* dXQ, int BH, int H, int NC, int G, int t0, int nsteps,
                                  cudaStream_t stream, unsigned* ready) {
  static bool attr_done_dev[64] = {};  // function attributes (and side streams) are per device
  bool& attr_done = *device_once(attr_done_dev);
  if (!attr_done) {
    TB_TRY(cudaFuncSetAttribute(bwd::ttt_mlp_bwd_q_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd::QS_TOTAL), "smem attr (q)");
    attr_done = true;
  }
  bwd::BwdQParams p{};
  p.ln_w = ln_w; p.ln_b = ln_b; p.slot = slot; p.dXQ = reinterpret_cast<__nv_bfloat16*>(dXQ);
  p.H = H; p.NC = NC; p.img_slots = G + 1; p.G = G; p.t0 = t0; p.ready = ready;
  dim3 grid(nsteps, BH);
  bwd::ttt_mlp_bwd_q_kernel<<<grid, 256, bwd::QS_TOTAL, stream>>>(tq, tdo, p);
  return cudaGetLastError();
}

}  // namespace tb
