// TTT-Linear forward scan for sm_100a.  Replaces the Triton kernel ttt/models/ssm/kernels/linear_forward.py:5-148
// (launched from ttt/models/ssm/linear_triton.py:96-131); arithmetic = ttt/models/ssm/ops/ttt_linear.py:8-56 in primal
// form (Z1bar = XQ.W1' + b1', kernels/linear_forward.py:128-134), LayerNorm eps 1e-8.
//
// CS = 16 is below tcgen05's M >= 64, so the GEMMs run transposed with the 64-wide OUTPUT feature dim on M, and TWO
// (batch,head) sequences are stacked on the 128 TMEM lanes of one CTA (the reference launches one Triton program per
// head and lights 48 SMs; here 24 CTAs do the same work with full-shape M=128 MMAs):
//   W1^T stack [128 = 2 seq x 64 f_out][64 f_in] fp32 is a persistent TMEM accumulator (+ a bf16 K-major operand copy)
//   D1 = W1b^T . [K_s0 | K_s1 | Q_s0 | Q_s1]^T  -> [128 x 64 token columns]; each row uses only its own sequence's columns
//   update: W1^T += G^T . K   with A = G (MN-major, 32 token rows x 2 blocks of 64; the other sequence's rows are zero)
// LayerNorm reduces over features = over TMEM lanes here, so Z1 goes through an fp32 smem transpose (padded rows) and is
// normalised by 64 token threads (one row each), exactly like the eager code.  Q side of step t-1 rides with K side of t.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ptx.cuh"
#include "recompute_ring.cuh"
#include "ttt_internal.h"

namespace tb {
namespace lin {

constexpr int CS = 16, F = 64, NT = 128;
constexpr int ZP = 66;  // fp32 transpose buffer row: two 32-column halves padded to 33 (bank-conflict free for the
                        // (row, half) thread pairs of the LayerNorm phase)
__device__ __forceinline__ int zidx(int row, int f) { return row * ZP + (f >> 5) * 33 + (f & 31); }

constexpr uint32_t SM_W1B = 0;                       // [128][64] bf16 K-major                   16 KB
constexpr uint32_t SM_TOK = 16384;                   // 2 slots x 64 rows: K_s0,K_s1,Q_s0,Q_s1   16 KB
constexpr uint32_t SM_V = SM_TOK + 16384;            // 2 slots x 32 rows: V_s0, V_s1             8 KB
constexpr uint32_t SM_GT = SM_V + 8192;              // G^T operand: 2 blocks x 32 token rows     8 KB
constexpr uint32_t SM_ZT = SM_GT + 8192;             // fp32 [64 token rows][66]                 16896 B
constexpr uint32_t SM_MISC = SM_ZT + 64 * ZP * 4;    // ln params of both sequences, barriers
constexpr uint32_t SM_TOTAL = SM_MISC + 2048;

constexpr uint32_t TM_W1 = 0, TM_D1 = 64;

struct LinParams {
  const __nv_bfloat16* last_eta;  // [B,H,NC,16]
  const float *ln_w, *ln_b;       // [H,64]
  const float *W1, *b1;           // [B,H,64,64], [B,H,64]
  float *W1c, *b1c;               // checkpoints [B,H,K,64,64], [B,H,K,64] (may be null)
  float *W1o, *b1o;               // final state (may be null)
  __nv_bfloat16* Out;             // [B,H,NC,16,64]
  int BH, H, NC, ckpt_group, K;
  // trajectory mode (backward recompute, ttt_linear_bwd.cu): run steps t0 .. t0+nsteps-1 (K side only) from the state
  // at W1 + bh*w_stride (b1 + bh*b_stride) and save the bf16 operand image of the state BEFORE step t0+i in record i and
  // the state after the last step in record nsteps (recompute_ring.cuh)
  long long w_stride, b_stride;
  int t0, nsteps, img_slots;
  LinearImages out;
};

template <bool kTraj>
__global__ void __launch_bounds__(NT, 1)
ttt_linear_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                      const __grid_constant__ CUtensorMap tmV, const LinParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int warp_u = uniform_warp_id();  // == warp, provably warp-uniform: single-thread issue blocks branch on it
  const int NC = kTraj ? p.nsteps : p.NC;  // steps this launch runs (trajectory mode: a window of the sequence)
  const int s_row = tid >> 6;            // which of the two stacked sequences this W1^T row belongs to
  const int fo = tid & 63;               // output feature of this row
  const int bh_row = 2 * blockIdx.x + s_row;
  const bool row_valid = bh_row < p.BH;  // odd BH: the second sequence of the last CTA is a dummy
  const uint32_t lane_addr = ((uint32_t)(warp * 32)) << 16;

  float* zt = reinterpret_cast<float*>(smem + SM_ZT);
  float* lnw = reinterpret_cast<float*>(smem + SM_MISC);  // [2][64]
  float* lnb = lnw + 128;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_MISC + 1024);
  uint64_t* tma_bar = bars;      // [2]
  uint64_t* mma_bar = bars + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 4);

  if (warp_u == 0 && elect_one()) {
    mbar_init(&tma_bar[0], 1);
    mbar_init(&tma_bar[1], 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV);
  }
  if (warp == 0) tmem_alloc<128>(tmem_ptr);
  {
    const int bhc = row_valid ? bh_row : 0;
    lnw[tid] = p.ln_w[(bhc % p.H) * 64 + fo];
    lnb[tid] = p.ln_b[(bhc % p.H) * 64 + fo];
  }
  // zero the token / V tiles (a dummy second sequence must contribute finite values to the stacked MMAs) and the G^T
  // operand (rows of the other sequence stay zero for the whole kernel)
  for (int i = tid; i < (SM_ZT - SM_TOK) / 16; i += NT) st_shared_v4(sbase + SM_TOK + 16 * i, 0, 0, 0, 0);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;

  // LayerNorm-phase roles (all 128 threads): token row = tid >> 1 (sequence ts, token tt: 0-15 K side, 16-31 Q side),
  // column half ch = tid & 1; the two threads of a row are adjacent lanes and exchange partial sums by shuffle.  Each
  // warp is uniformly K side or Q side: warp 0 = seq0 K, 1 = seq0 Q, 2 = seq1 K, 3 = seq1 Q.
  const int trow_id = tid >> 1, ch = tid & 1;
  const int ts = trow_id >> 5, tt = trow_id & 31;
  const int bh_tok = 2 * blockIdx.x + ts;
  const bool tok_valid = bh_tok < p.BH;

  auto issue_loads = [&](int it, int slot) {  // K_it, V_it (if it < NC) and Q_{it-1} (if it > 0) of both sequences
    uint32_t bytes = 0;
    for (int s = 0; s < 2; ++s) {
      if (2 * (int)blockIdx.x + s >= p.BH) continue;
      if (it < NC) bytes += 4096;
      if (!kTraj && it > 0) bytes += 2048;
    }
    mbar_expect_tx(&tma_bar[slot], bytes);
    for (int s = 0; s < 2; ++s) {
      const int bh = 2 * blockIdx.x + s;
      if (bh >= p.BH) continue;
      const int row0 = (bh * p.NC + (kTraj ? p.t0 : 0)) * CS;
      if (it < NC) {
        tma_load_2d(smem + SM_TOK + slot * 8192 + s * 2048, &tmK, 0, row0 + it * CS, &tma_bar[slot]);
        tma_load_2d(smem + SM_V + slot * 4096 + s * 2048, &tmV, 0, row0 + it * CS, &tma_bar[slot]);
      }
      if (!kTraj && it > 0) tma_load_2d(smem + SM_TOK + slot * 8192 + 4096 + s * 2048, &tmQ, 0, row0 + (it - 1) * CS, &tma_bar[slot]);
    }
  };
  if (warp_u == 0 && elect_one()) issue_loads(0, 0);

  // ---- initial state -> TMEM accumulator + bf16 operand copy (+ checkpoint 0)
  float b1r = row_valid ? p.b1[(size_t)bh_row * p.b_stride + fo] : 0.f;
  {
    const float* W1g = p.W1 + (size_t)(row_valid ? bh_row : 0) * p.w_stride;
    uint32_t v[32];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = row_valid ? __float_as_uint(W1g[(size_t)(32 * c + i) * F + fo]) : 0u;
      tmem_st32(tmem + lane_addr + TM_W1 + 32 * c, v);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        st_shared_v4(sbase + SM_W1B + sw128_off(tid, 4 * c + q),
                     pack_bf16(__uint_as_float(v[8 * q]), __uint_as_float(v[8 * q + 1])),
                     pack_bf16(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3])),
                     pack_bf16(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5])),
                     pack_bf16(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7])));
      if (p.W1c && row_valid)
#pragma unroll
        for (int i = 0; i < 32; ++i) p.W1c[((size_t)bh_row * p.K) * F * F + (size_t)(32 * c + i) * F + fo] = __uint_as_float(v[i]);
    }
    if (p.b1c && row_valid) p.b1c[((size_t)bh_row * p.K) * F + fo] = b1r;
    tc_wait_st();
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();

  constexpr uint32_t IDESC_1 = make_idesc_bf16(128, 64, false, false);  // D1: A K-major, B K-major
  constexpr uint32_t IDESC_U = make_idesc_bf16(128, 64, true, true);    // update: A MN-major (2 blocks), B MN-major
  uint32_t mma_phase = 0;

  for (int it = 0; it <= NC; ++it) {
    const int slot = it & 1;
    const bool has_k = it < NC, has_q = !kTraj && it > 0;
    const uint32_t tok = sbase + SM_TOK + slot * 8192;
    const uint32_t vt = sbase + SM_V + slot * 4096;
    float eta_i = 0.f;
    if (has_k && tok_valid && tt < 16)  // both threads of the row
      eta_i = __bfloat162float(p.last_eta[((size_t)bh_tok * p.NC + (kTraj ? p.t0 : 0) + it) * CS + tt]);
    if (kTraj) {  // image of the state before this step (record it; the last pass, it == nsteps, saves the final state)
      p.out.image_b1(blockIdx.x, p.img_slots, it)[tid] = b1r;
      if (warp_u == 0 && elect_one()) {
        bulk_store_1d(p.out.image(blockIdx.x, p.img_slots, it), smem + SM_W1B, kLinImageBytes);
        bulk_commit();
      }
      if (!has_k) break;
    }

    mbar_wait(&tma_bar[slot], (it >> 1) & 1);
    if (warp_u == 0 && (it < NC) && elect_one()) issue_loads(it + 1, slot ^ 1);

    // ---- MMA-1: D1 = W1b^T . TOK^T   (M=128, N=64 token columns, K=64)
    if (warp_u == 0 && elect_one()) {
      tc_fence_after();
      const uint64_t da = make_desc_sw128(sbase + SM_W1B, 16, 1024);
      const uint64_t db = make_desc_sw128(tok, 16, 1024);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_ss(tmem + TM_D1, desc_advance(da, 32 * k), desc_advance(db, 32 * k), IDESC_1, k > 0);
      tc_commit(mma_bar);
    }
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();

    // ---- EW-A: this row's own-sequence columns (+ b1) -> fp32 transpose buffer zt[(s*32 + token)][f_out]
    {
      uint32_t vk[16], vq[16];
      tmem_ld16(tmem + lane_addr + TM_D1 + 16 * s_row, vk);
      tmem_ld16(tmem + lane_addr + TM_D1 + 32 + 16 * s_row, vq);
      tc_wait_ld();
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        zt[zidx(s_row * 32 + i, fo)] = __uint_as_float(vk[i]) + b1r;
        zt[zidx(s_row * 32 + 16 + i, fo)] = __uint_as_float(vq[i]) + b1r;
      }
    }
    tc_fence_before();
    __syncthreads();

    // ---- EW-B: LayerNorm per token row: 2 threads per row (32 columns each), all 4 warps
    if (tok_valid && ((tt < 16) ? has_k : has_q)) {
      float z[32];
      float* zr = zt + (ts * 32 + tt) * ZP + ch * 33;
      float a1 = 0.f, a2 = 0.f;
#pragma unroll
      for (int f = 0; f < 32; ++f) { z[f] = zr[f]; a1 += z[f]; a2 = fmaf(z[f], z[f], a2); }
      a1 += __shfl_xor_sync(0xffffffffu, a1, 1);
      a2 += __shfl_xor_sync(0xffffffffu, a2, 1);
      const float mu = a1 * (1.f / 64.f);
      const float rstd = rsqrtf(fmaxf(a2 * (1.f / 64.f) - mu * mu, 0.f) + 1e-8f);
      const float* gw = lnw + ts * 64 + 32 * ch;
      const float* gb = lnb + ts * 64 + 32 * ch;
      if (tt < 16) {
        const int r = 16 * ts + tt;  // row of K in the token tile and of V in the V tile
        float g[32];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t kk[4], vv[4];
          ld_shared_v4(tok + sw128_off(r, 4 * ch + c), kk[0], kk[1], kk[2], kk[3]);
          ld_shared_v4(vt + sw128_off(r, 4 * ch + c), vv[0], vv[1], vv[2], vv[3]);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int f = 8 * c + 2 * e;
            z[f] = (z[f] - mu) * rstd; z[f + 1] = (z[f + 1] - mu) * rstd;
            g[f] = (fmaf(gw[f], z[f], gb[f]) - (bf16_lo(vv[e]) - bf16_lo(kk[e]))) * gw[f];
            g[f + 1] = (fmaf(gw[f + 1], z[f + 1], gb[f + 1]) - (bf16_hi(vv[e]) - bf16_hi(kk[e]))) * gw[f + 1];
            s1 += g[f] + g[f + 1];
            s2 = fmaf(g[f], z[f], fmaf(g[f + 1], z[f + 1], s2));
          }
        }
        s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
        s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
        const float sc = -eta_i * rstd * (1.f / 64.f);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int f = 8 * c + 2 * e;
            const float d0 = (fmaf(64.f, g[f], -s1) - z[f] * s2) * sc;
            const float d1 = (fmaf(64.f, g[f + 1], -s1) - z[f + 1] * s2) * sc;
            zr[f] = d0; zr[f + 1] = d1;   // fp32 G = -eta * gradZ1 for the b1 column sums
            o[e] = pack_bf16(d0, d1);
          }
          st_shared_v4(sbase + SM_GT + ts * 4096 + sw128_off(r, 4 * ch + c), o[0], o[1], o[2], o[3]);
        }
      } else {
        const int tq = tt - 16;
        const int r = 32 + 16 * ts + tq;  // row of Q_{it-1} in the token tile
        __nv_bfloat16* og = p.Out + (((size_t)bh_tok * NC + (it - 1)) * CS + tq) * F + 32 * ch;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t qq[4], o[4];
          ld_shared_v4(tok + sw128_off(r, 4 * ch + c), qq[0], qq[1], qq[2], qq[3]);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int f = 8 * c + 2 * e;
            o[e] = pack_bf16(bf16_lo(qq[e]) + fmaf(gw[f], (z[f] - mu) * rstd, gb[f]),
                             bf16_hi(qq[e]) + fmaf(gw[f + 1], (z[f + 1] - mu) * rstd, gb[f + 1]));
          }
          *reinterpret_cast<uint4*>(og + 8 * c) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    if (!has_k) break;
    fence_proxy_async();
    __syncthreads();

    // ---- MMA-U: W1^T += G^T . K   (A MN-major: 32 token rows x 2 blocks of 64 f_out; B = K rows of the token tile)
    if (warp_u == 0 && elect_one()) {
      if (kTraj) bulk_wait_read<0>();  // the image store must have read W1b before the epilogue below rewrites it
      tc_fence_after();
      const uint64_t da = make_desc_sw128(sbase + SM_GT, 4096, 1024);
      const uint64_t db = make_desc_sw128(tok, 1024, 1024);
#pragma unroll
      for (int k = 0; k < 2; ++k) umma_ss(tmem + TM_W1, desc_advance(da, 2048 * k), desc_advance(db, 2048 * k), IDESC_U, 1);
      tc_commit(mma_bar);
    }
    // ---- EW-C (overlaps the MMA): b1 += column sums of G over this sequence's 16 tokens
    {
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) acc += zt[zidx(s_row * 32 + i, fo)];
      b1r += acc;
    }
    mbar_wait(mma_bar, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();
    {
      const int nstep = it + 1;
      const bool ck = !kTraj && p.W1c && row_valid && nstep < NC && (nstep % p.ckpt_group == 0);
      const bool fin = !kTraj && p.W1o && row_valid && nstep == NC;
      const size_t kidx = ck ? ((size_t)bh_row * p.K + nstep / p.ckpt_group) : 0;
      uint32_t v[32];
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        tmem_ld32(tmem + lane_addr + TM_W1 + 32 * c, v);
        tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 4; ++q)
          st_shared_v4(sbase + SM_W1B + sw128_off(tid, 4 * c + q),
                       pack_bf16(__uint_as_float(v[8 * q]), __uint_as_float(v[8 * q + 1])),
                       pack_bf16(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3])),
                       pack_bf16(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5])),
                       pack_bf16(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7])));
        if (ck)
#pragma unroll
          for (int i = 0; i < 32; ++i) p.W1c[kidx * F * F + (size_t)(32 * c + i) * F + fo] = __uint_as_float(v[i]);
        if (fin)
#pragma unroll
          for (int i = 0; i < 32; ++i) p.W1o[(size_t)bh_row * F * F + (size_t)(32 * c + i) * F + fo] = __uint_as_float(v[i]);
      }
      if (ck) p.b1c[kidx * F + fo] = b1r;
      if (fin) p.b1o[(size_t)bh_row * F + fo] = b1r;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
  }

  if (kTraj && warp_u == 0 && elect_one()) bulk_wait<0>();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<128>(tmem);
}

}  // namespace lin

cudaError_t launch_linear_forward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                  const float* ln_b, const float* W1, const float* b1, float* W1c, float* b1c,
                                  float* W1o, float* b1o, void* Out, int B, int H, int NC, int ckpt_group,
                                  cudaStream_t stream) {
  if (B <= 0 || H <= 0 || NC <= 0 || ckpt_group <= 0) { g_where = "bad sizes"; return cudaErrorInvalidValue; }
  const uint64_t rows = (uint64_t)B * H * NC * lin::CS;
  if (rows > 0x7FFFFFFFull) { g_where = "too many rows"; return cudaErrorInvalidValue; }
  CUtensorMap tq, tk, tv;
  if (make_token_tmap_box(&tq, XQ, rows, 16) || make_token_tmap_box(&tk, XK, rows, 16) || make_token_tmap_box(&tv, XV, rows, 16))
    return cudaErrorInvalidValue;
  lin::LinParams p{};
  p.last_eta = reinterpret_cast<const __nv_bfloat16*>(last_eta);
  p.ln_w = ln_w; p.ln_b = ln_b; p.W1 = W1; p.b1 = b1; p.W1c = W1c; p.b1c = b1c; p.W1o = W1o; p.b1o = b1o;
  p.Out = reinterpret_cast<__nv_bfloat16*>(Out);
  p.BH = B * H; p.H = H; p.NC = NC; p.ckpt_group = ckpt_group; p.K = (NC + ckpt_group - 1) / ckpt_group;
  p.w_stride = lin::F * lin::F; p.b_stride = lin::F;
  static bool attr_done_dev[64] = {};  // function attributes (and side streams) are per device
  bool& attr_done = *device_once(attr_done_dev);
  if (!attr_done) {
    TB_TRY(cudaFuncSetAttribute(lin::ttt_linear_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lin::SM_TOTAL), "smem attr");
    attr_done = true;
  }
  g_where = "linear forward launch";
  lin::ttt_linear_fwd_kernel<false><<<(p.BH + 1) / 2, lin::NT, lin::SM_TOTAL, stream>>>(tq, tk, tv, p);
  return cudaGetLastError();
}

// Backward recompute: steps t0 .. t0+nsteps-1 from the checkpointed state (W1s + bh*w_stride, b1s + bh*b_stride), saving
// nsteps+1 operand images (see LinParams).  Used by launch_linear_backward (ttt_linear_bwd.cu).
cudaError_t launch_linear_trajectory(const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                     const float* ln_b, const float* W1s, const float* b1s, long long w_stride,
                                     long long b_stride, const LinearImages& out, int img_slots, int B, int H, int NC,
                                     int t0, int nsteps, cudaStream_t stream) {
  if (nsteps <= 0 || nsteps + 1 > img_slots || t0 < 0 || t0 + nsteps > NC) { g_where = "bad trajectory window"; return cudaErrorInvalidValue; }
  const uint64_t rows = (uint64_t)B * H * NC * lin::CS;
  CUtensorMap tk, tv;
  if (make_token_tmap_box(&tk, XK, rows, 16) || make_token_tmap_box(&tv, XV, rows, 16)) return cudaErrorInvalidValue;
  lin::LinParams p{};
  p.last_eta = reinterpret_cast<const __nv_bfloat16*>(last_eta);
  p.ln_w = ln_w; p.ln_b = ln_b; p.W1 = W1s; p.b1 = b1s; p.w_stride = w_stride; p.b_stride = b_stride;
  p.BH = B * H; p.H = H; p.NC = NC; p.ckpt_group = 1; p.K = 1;
  p.t0 = t0; p.nsteps = nsteps; p.img_slots = img_slots; p.out = out;
  static bool attr_done_dev[64] = {};  // function attributes (and side streams) are per device
  bool& attr_done = *device_once(attr_done_dev);
  if (!attr_done) {
    TB_TRY(cudaFuncSetAttribute(lin::ttt_linear_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lin::SM_TOTAL), "smem attr");
    attr_done = true;
  }
  g_where = "linear trajectory launch";
  lin::ttt_linear_fwd_kernel<true><<<(p.BH + 1) / 2, lin::NT, lin::SM_TOTAL, stream>>>(tk, tk, tv, p);
  return cudaGetLastError();
}

}  // namespace tb
