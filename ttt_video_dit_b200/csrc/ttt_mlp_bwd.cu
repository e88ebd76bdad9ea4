// TTT-MLP backward for sm_100a.  Replaces ttt-tk/kernels/ttt_backward/ttt.cu:179-1917 (bwd_ttt_mlp_ker / ttt_backward).
//
// Structure (differs from the reference on purpose, SURVEY 7 "Backward memory traffic"): per checkpoint group g, in
// reverse order, three kernels on three streams (DESIGN.md section 4):
//   1. trajectory  (csrc/ttt_mlp_traj.cu): re-runs the K side of the group's steps from the fp32 checkpoint and stores only
//      the bf16 operand images of each state W_t (64 KB/step) -- the reference spills 16 intermediates per step
//      (~338 KB/step, SURVEY 8a row a7);
//   2. Q side      (csrc/ttt_mlp_bwd_q.cu): the backward of the output half of every step, which does not depend on the
//      carried state gradient: one CTA per (sequence, step) on the SMs the sequential kernels leave idle; emits dQ and
//      the factor tiles of its contribution to dW1 / dW2;
//   3. K side      (this file): the sequential chain.  Walks t = t_hi .. t_lo; iteration t recomputes the K side of step t
//      from the image of W_t, applies the closed-form backward (SURVEY appendix B = ttt-tk/kernels/ttt_backward/
//      matching.py:173-342) and adds the Q-side factor tiles of step t with two accumulate-MMAs.  In persistent mode one
//      launch walks every group and hand-shakes with the other two kernels through device-side counters.
// dW1^T, dW2 (grad w.r.t. the carried state) are persistent fp32 TMEM accumulators; between launches (per-group mode) they
// live in a small fp32 scratch.  Same "hidden units on TMEM lanes" layout as the forward; all tiles are SW128 row tiles.
// The hidden-lane element-wise phases use packed fp32 pairs (FFMA2, ptx.cuh); the token phases are scalar (measured).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "bwd_common.cuh"
#include "ptx.cuh"
#include "recompute_ring.cuh"
#include "ttt_internal.h"

namespace tb {
namespace bwd {

constexpr int CS = 64, F = 64, HID = 256, NT = 256;

// ---- shared memory map (bytes); total = 232448 = the 227 KB per-CTA maximum
constexpr uint32_t SM_W2I = 0;         // W2 image of W_t                     [256][64] bf16
constexpr uint32_t SM_HS = 32768;      // 4 hidden-lane tile slots of 32 KB (roles rotate, see kernel)
constexpr uint32_t SM_TK = 163840;     // K_t   [64][64]
constexpr uint32_t SM_TQ = 172032;     // Q_{t-1}
constexpr uint32_t SM_TV = 180224;     // V_t
constexpr uint32_t SM_TDO = 188416;    // dOut_{t-1}
constexpr uint32_t SM_TT0 = 196608;    // dZ2 (K side) / dZbar2 (Q side)
constexpr uint32_t SM_TT1 = 204800;    // gradZ2
constexpr uint32_t SM_TT2 = 212992;    // -eta*gradZ2
constexpr uint32_t SM_MISC = 221184;   // small fp32 vectors, barriers (2560 B)
constexpr uint32_t SM_XB = SM_MISC + 2560;  // token-phase exchange buffers: float4[4][64], float2[4][64], float[4][64]
constexpr uint32_t SM_TOTAL = SM_XB + 7680;  // 231424 (+512: second-row-half accumulators of d gamma / d beta)
static_assert(SM_TOTAL <= 231424, "smem budget: 227 KB minus the 1 KB alignment slack of the dynamic window");

// ---- TMEM columns
constexpr uint32_t TM_DW1 = 0;    // dW1^T accumulator, + 64*h
constexpr uint32_t TM_DW2 = 128;  // dW2   accumulator, + 64*h
constexpr uint32_t TM_S0 = 256, TM_S1 = 320, TM_S2 = 384, TM_S3 = 448;  // working slots of 64 columns

struct BwdParams {
  const __nv_bfloat16* last_eta;  // [B,H,NC,64]
  const float *ln_w, *ln_b;       // [H,64]
  MlpSlot ring[kRingSlots];  // recompute buffers (recompute_ring.cuh); inside a slot, step t is local index t - g*G
  float *dW1s, *dW2s, *db1s, *db2s;  // carried state gradient, fp32: [BH][256][64] x2, [BH][256], [BH][64]
  uint8_t* x2spill;                  // [BH][32 KB]
  int G, K;                          // steps per checkpoint group, number of groups
  __nv_bfloat16 *dXQ, *dXK, *dXV, *dEta;  // outputs
  float *dlnw, *dlnb;                     // [BH][64], accumulated launch after launch, one writer per element (pre-zeroed by the host)
  float *dW1, *db1, *dW2, *db2;           // final gradient w.r.t. the initial state (written when the launch ends at step 0)
  int H, NC, img_slots;
  int t_hi, t_lo;      // iterations t_hi..t_lo (descending).  Persistent mode: the whole scan in ONE launch (NC-1 .. 0)
  int first;           // 1: start from zero state gradient, 0: load it from the scratch
  // Persistent mode (both non-null): device-side hand-shake with the recompute kernels running on other SMs.
  //   ready[u * BH + bh] counts the Q-side CTAs of unit u, sequence bh, that have finished (the unit's images are complete
  //   before its Q-side kernel starts); the K-side CTA waits for the unit's step count before touching the unit's buffers.
  //   done[u * BH + bh] is set by the K-side CTA after its last access to unit u: the trajectory kernel of unit
  //   u + kRingSlots (same ring slot) waits for it before overwriting.
  const unsigned* ready;
  unsigned* done;
  unsigned* dbg;       // phase-timing buffer (debug builds)
  int dbg_group;       // group (t_lo / G) whose observer phase times are dumped
};

// out of line: the wait sits in the step loop, whose code size the instruction cache decides (DESIGN.md section 4)
static __device__ __noinline__ void wait_ready(const unsigned* flag, unsigned want) { wait_flag<256>(flag, want); }

__global__ void __launch_bounds__(NT, 1)
ttt_mlp_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warp_u = uniform_warp_id();  // == warp, provably warp-uniform: single-thread issue blocks branch on it
  const int bh = blockIdx.x, head = bh % p.H;
  const int half = warp >> 2;
  const uint32_t lane_addr = ((uint32_t)((warp & 3) * 32)) << 16;
  const int j = tid;
  TICK_DECL(22, 224)
#ifdef TTT_PHASE_TIMING
  const long long tick_t0_64 = clock64();
  unsigned long long tick_g0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tick_g0));
#endif

  float* lnw = reinterpret_cast<float*>(smem + SM_MISC);  // [64]
  float* lnb = lnw + 64;
  float* b2t = lnb + 64;      // b2 of W_t
  float* db2c = b2t + 64;     // d b2 carried (grad w.r.t. b2 after step t; updated in place during the iteration)
  float* etas = db2c + 64;    // -eta of step t (every use multiplies by -eta)
  // Reductions over token rows / hidden lanes are laid out so that every shared-memory word has exactly ONE writer per
  // step (no atomics): fp32 addition is not associative, and an unordered pair of adds onto a running sum would make the
  // whole backward bit-irreproducible (d b2 feeds every earlier step).  Row halves (warp & 1) own separate accumulators.
  float* db2h = etas + 64;    // d b2 contributions of token rows 32-63 of the current step (merged at the loop top)
  float* dgam = db2h + 64;    // d gamma / d beta accumulated over the whole launch, token rows 0-31 (+ Q-side partials)
  float* dbet = dgam + 64;
  float* dgam2 = reinterpret_cast<float*>(smem + SM_XB + 7168);  // ... token rows 32-63
  float* dbet2 = dgam2 + 64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_MISC + 2048);
  uint64_t* mma_bar = bars;       // tcgen05.commit
  uint64_t* bar_kv = bars + 1;    // K_t, V_t tiles
  uint64_t* bar_qd = bars + 2;    // Q_{t-1}, dO_{t-1} tiles
  uint64_t* bar_w1 = bars + 3;    // W1 image at iteration start
  uint64_t* bar_w1r = bars + 4;   // W1 image reload (for dK / dQ GEMMs)
  uint64_t* bar_w2 = bars + 5;    // W2 image
  uint64_t* bar_x2 = bars + 6;    // X2 tile reload
  uint64_t* bar_aux = bars + 7;   // completion of the early dW2 accumulations (frees two tile slots)
  uint64_t* bar_xb = bars + 8;    // Q-side Xbar2^T factor tile
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 12);
  float4* xA = reinterpret_cast<float4*>(smem + SM_XB);          // [4][64]
  float2* xB = reinterpret_cast<float2*>(smem + SM_XB + 4096);   // [4][64]
  float* epart = reinterpret_cast<float*>(smem + SM_XB + 6144);  // [4][64]
  // xA carries float2 payloads in .x/.y; the .z/.w words hold the 8 per-warp partial sums of the d eta reduction over the
  // hidden lanes (one word per (warp, token)), written in A5/A6 and read in A8
  float* esum8 = reinterpret_cast<float*>(smem + SM_XB);
  // token-phase mapping: thread <-> (row trow, column quarter cq); row r is read from TMEM lane r (warps with
  // (warp&3) < 2) or from its duplicate at lane 64+r (the others) -- both inside this warp's own lane quarter.
  const int trow = 32 * (warp & 1) + lane;
  const int cq = 2 * (warp >> 2) + ((warp >> 1) & 1);
  const int c0 = 16 * cq;

  if (warp_u == 0 && elect_one()) {
    for (int i = 0; i < 9; ++i) mbar_init(&bars[i], 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV);
  }
  if (warp == 0) tmem_alloc<512>(tmem_ptr);
  if (tid < 64) {
    lnw[tid] = p.ln_w[head * 64 + tid];
    lnb[tid] = p.ln_b[head * 64 + tid];
    db2c[tid] = p.first ? 0.f : p.db2s[(size_t)bh * 64 + tid];
    db2h[tid] = 0.f;
    dgam[tid] = 0.f; dbet[tid] = 0.f; dgam2[tid] = 0.f; dbet2[tid] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;

  const size_t row_bh = (size_t)bh * p.NC * CS;  // token row of step 0 of this sequence
  // ring addressing of the per-step recompute data (see BwdParams).  The pointers of the current step and of the next one
  // (t - 1, whose loads are issued during step t) are kept in registers and advanced once per iteration: no divisions in
  // the step loop.
  struct StepIdx { int r, l; };  // ring slot and local index inside it
  auto step_idx = [&](int t) { const int g = t / p.G; return StepIdx{ring_slot(unit_of_group(g, p.K)), t - group_begin(g, p.G)}; };
  auto step_back = [&](StepIdx& si) {  // index of the step before the one si points at
    // crossing into the previous checkpoint group = the next unit: next ring slot, last local index (every group below the
    // last one is full)
    if (si.l == 0) { si.r = (si.r + 1) % kRingSlots; si.l = p.G - 1; }
    else --si.l;
  };
  auto img_at = [&](StepIdx si) { return p.ring[si.r].image(bh, p.img_slots, si.l); };
  auto qt_at = [&](StepIdx si) { return p.ring[si.r].factors(bh, p.G, si.l); };
  auto b1_at = [&](StepIdx si) { return p.ring[si.r].image_b1(bh, p.img_slots, si.l); };
  auto b2_at = [&](StepIdx si) { return p.ring[si.r].image_b2(bh, p.img_slots, si.l); };
  auto q1_at = [&](StepIdx si) { return p.ring[si.r].factor_b1(bh, p.G, si.l); };
  auto q2_at = [&](StepIdx si) { return p.ring[si.r].factor_vec(bh, p.G, si.l); };
  StepIdx cur = step_idx(p.t_hi), nxt = cur;  // nxt: step t - 1 (valid while t > t_lo)
  if (p.t_hi > p.t_lo) step_back(nxt);
  // persistent mode: before the first access to the buffers of the unit that holds step t
  auto wait_unit_of = [&](int t) {
    if (p.ready == nullptr) return;
    const int g = t / p.G, u = unit_of_group(g, p.K);
    const int steps = min(p.NC, group_begin(g + 1, p.G)) - group_begin(g, p.G);
    wait_ready(p.ready + (size_t)u * gridDim.x + bh, (unsigned)steps);
  };
  // slot roles (byte offsets of the four 32 KB hidden-lane slots); they rotate every iteration
  uint32_t sW1 = SM_HS, sA = SM_HS + 32768, sB = SM_HS + 65536, sC = SM_HS + 98304;
  uint32_t mma_phase = 0, ph_kv = 0, ph_qd = 0, ph_w1 = 0, ph_w1r = 0, ph_w2 = 0, ph_x2 = 0, ph_aux = 0, ph_xb = 0;

  // Loads that feed iteration t: Q_t tile + the Q-side factor tiles of step t.  Thread 0 only.
  int tcur = p.t_hi;  // the step `cur` points at (load helpers take t = tcur or tcur - 1)
  auto load_xb = [&](int t, uint32_t xs) {  // Xbar2^T factor tile of step t
    mbar_expect_tx(bar_xb, 32768);
    bulk_load_1d(smem + xs, qt_at(t == tcur ? cur : nxt), 32768, bar_xb);
  };
  auto load_q_rest = [&](int t, uint32_t zs) {  // Q_t tile, dZbar1^T -> slot zs, dZbar2 -> TT0
    const uint8_t* src = qt_at(t == tcur ? cur : nxt);
    mbar_expect_tx(bar_qd, 8192 + 32768 + 8192);
    tma_load_2d(smem + SM_TQ, &tmQ, 0, (int)(row_bh + (size_t)t * CS), bar_qd);
    bulk_load_1d(smem + zs, src + kFactorDZbar1T, 32768, bar_qd);
    bulk_load_1d(smem + SM_TT0, src + kFactorDZbar2, 8192, bar_qd);
  };
  // first iteration's loads, issued before the carried gradient is read so that both latencies overlap
  wait_unit_of(p.t_hi);
  if (warp_u == 0 && elect_one()) {
    const int t = p.t_hi;
    const uint8_t* im = img_at(cur);
    mbar_expect_tx(bar_w1, 32768);
    bulk_load_1d(smem + sW1, im, 32768, bar_w1);
    mbar_expect_tx(bar_w2, 32768);
    bulk_load_1d(smem + SM_W2I, im + kImageW2, 32768, bar_w2);
    mbar_expect_tx(bar_kv, 16384);
    tma_load_2d(smem + SM_TK, &tmK, 0, (int)(row_bh + (size_t)t * CS), bar_kv);
    tma_load_2d(smem + SM_TV, &tmV, 0, (int)(row_bh + (size_t)t * CS), bar_kv);
    load_xb(t, sA);
    load_q_rest(t, sB);
  }
  // ---- carried state gradient -> TMEM
  float db1r = p.first ? 0.f : p.db1s[(size_t)bh * HID + j];
  {
    uint32_t v[32];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      if (p.first) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = 0u;
        tmem_st32(tmem + lane_addr + TM_DW1 + 64 * half + 32 * c, v);
        tmem_st32(tmem + lane_addr + TM_DW2 + 64 * half + 32 * c, v);
      } else {
        const uint4* s1 = reinterpret_cast<const uint4*>(p.dW1s + ((size_t)bh * HID + j) * F + 32 * c);
        const uint4* s2 = reinterpret_cast<const uint4*>(p.dW2s + ((size_t)bh * HID + j) * F + 32 * c);
#pragma unroll
        for (int i = 0; i < 8; ++i) { const uint4 q = s1[i]; v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w; }
        tmem_st32(tmem + lane_addr + TM_DW1 + 64 * half + 32 * c, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) { const uint4 q = s2[i]; v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w; }
        tmem_st32(tmem + lane_addr + TM_DW2 + 64 * half + 32 * c, v);
      }
    }
    tc_wait_st();
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();

  uint32_t g1p[32], g2p[32];  // packed bf16: gelu'(Z1) (later gelu'(Zbar1)), gelu''(Z1) (later term2)

  float nb1 = b1_at(cur)[j], nb2 = 0.f;
  float nq1 = q1_at(cur)[j], nq2 = 0.f, nqg = 0.f, nqb = 0.f;
  unsigned short neta = 0;
  if (tid < 64) {
    nb2 = b2_at(cur)[tid];
    const float* q2 = q2_at(cur);
    nq2 = q2[kFactorDb2 + tid]; nqg = q2[kFactorDgamma + tid]; nqb = q2[kFactorDbeta + tid];
    if (p.t_hi < p.NC) neta = reinterpret_cast<const unsigned short*>(p.last_eta)[row_bh + (size_t)p.t_hi * CS + tid];
  }
  TICK(14);  // prologue
  for (int t = p.t_hi; t >= p.t_lo; --t) {
    const bool has_k = true;
    // per-iteration small vectors were prefetched into registers during the previous iteration (nb1/nb2/neta)
    const float b1t = nb1;
    const float q1t = nq1;
    if (tid < 64) {
      b2t[tid] = nb2;
      etas[tid] = -__uint_as_float((uint32_t)neta << 16);
      // merge the second row half of the previous step, then the Q-side contribution of step t (state after step t)
      db2c[tid] = (db2c[tid] + db2h[tid]) + nq2;
      db2h[tid] = 0.f;
      dgam[tid] += nqg;  // Q-side (output LayerNorm) part of d gamma / d beta of step t
      dbet[tid] += nqb;
    }
    db1r += q1t;         // ... and to d b1
    if (t > p.t_lo) {  // prefetch for iteration t-1
      if (t % p.G == 0) wait_unit_of(t - 1);  // step t-1 opens the next unit (persistent mode): its recompute must be complete
      nb1 = b1_at(nxt)[j];
      nq1 = q1_at(nxt)[j];
      if (tid < 64) {
        nb2 = b2_at(nxt)[tid];
        const float* q2 = q2_at(nxt);
        nq2 = q2[kFactorDb2 + tid]; nqg = q2[kFactorDgamma + tid]; nqb = q2[kFactorDbeta + tid];
        neta = reinterpret_cast<const unsigned short*>(p.last_eta)[row_bh + (size_t)(t - 1) * CS + tid];
      }
    }
    mbar_wait(bar_w1, ph_w1); ph_w1 ^= 1;
    mbar_wait(bar_w2, ph_w2); ph_w2 ^= 1;
    mbar_wait(bar_kv, ph_kv); ph_kv ^= 1;
    __syncthreads();  // b2t / etas visible
      TICK(0);
#ifdef TTT_PHASE_TIMING
    if (p.dbg && tid == 0 && blockIdx.x == 0 && t < 4000) {  // wall-clock stamp of every step (block 0)
      unsigned long long gs;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gs));
      p.dbg[4096 + t] = (unsigned)gs;
    }
#endif

    if (has_k) {
      // ===== A1 MMA: R1 = W1 . K^T -> (S0,S1)
      if (warp_u == 0 && elect_one()) {
        tc_fence_after();
        mma_hid(tmem + TM_S0, tmem + TM_S1, sbase + sW1, sbase + SM_TK, false, 64, false);
        tc_commit(mma_bar);
      }
      MMA_WAIT();
      TICK(2);
      // ===== A2 [H]: Z1 -> X2 tile (sC), gelu', gelu''
      {
        const uint32_t src = tmem + lane_addr + (half ? TM_S1 : TM_S0);
        const f32x2 B1 = pk2(b1t);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          float v[32];
          tmem_ld32(src + 32 * c, reinterpret_cast<uint32_t*>(v));
          tc_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; i += 2) {  // two tokens per instruction (FFMA2)
            f32x2 x, a, e;
            gelu3x2(add2(pk2(v[i], v[i + 1]), B1), x, a, e);
            up2(x, v[i], v[i + 1]);
            g1p[16 * c + i / 2] = pack_bf16(a);
            g2p[16 * c + i / 2] = pack_bf16(e);
          }
          st_row32(sbase + sC, j, 4 * c, v);
        }
      }
      PHASE_SYNC();
      TICK(3);
      mbar_wait(bar_qd, ph_qd); ph_qd ^= 1;
      mbar_wait(bar_xb, ph_xb); ph_xb ^= 1;
      // ===== apply the Q-side contribution of step t to the carried gradient (outer products of the factor tiles written
      //       by ttt_mlp_bwd_q_kernel):  dW2 += Xbar2^T dZbar2 ;  dW1^T += dZbar1^T Q
      if (warp_u == 0 && elect_one()) {
        tc_fence_after();
        mma_hid(tmem + TM_DW2, tmem + TM_DW2 + 64, sbase + sA, sbase + SM_TT0, true, 64, true);
        mma_hid(tmem + TM_DW1, tmem + TM_DW1 + 64, sbase + sB, sbase + SM_TQ, true, 64, true);
        tc_commit(mma_bar);
      }
      MMA_WAIT();

      // ===== A0 [H]: bf16 copies of the carried gradient accumulators: CW1 -> sA, CW2 -> sB
      {
        float v[32];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          tmem_ld32(tmem + lane_addr + TM_DW1 + 64 * half + 32 * c, reinterpret_cast<uint32_t*>(v));
          tc_wait_ld();
          st_row32(sbase + sA, j, 4 * c, v);
          tmem_ld32(tmem + lane_addr + TM_DW2 + 64 * half + 32 * c, reinterpret_cast<uint32_t*>(v));
          tc_wait_ld();
          st_row32(sbase + sB, j, 4 * c, v);
        }
      }
      PHASE_SYNC();
      TICK(1);
      // ===== A3 MMA: R2: Z2 = X2 . W2 -> S2 ; B5: acc5 = X2 . CW2 -> S3
      if (warp_u == 0 && elect_one()) {
        tc_fence_after();
        mma_tok(tmem + TM_S2, sbase + sC, sbase + SM_W2I, false);
        mma_tok(tmem + TM_S3, sbase + sC, sbase + sB, false);
        tc_commit(mma_bar);
      }
      MMA_WAIT();
      TICK(4);
      // spill the X2 tile to L2 (needed again by the dW2 += X2^T dZ2 GEMM at the end of the K side)
      if (warp_u == 0 && elect_one()) {
        bulk_store_1d(p.x2spill + (size_t)bh * kX2SpillBytes, smem + sC, 32768);
        bulk_commit();
      }
      // ===== A4 [T] (all warps; thread = (row, 16 columns)): LN stats of Z2, gradZ2 -> TT1, -eta*gradZ2 -> TT2,
      //       dg2p = -eta(acc5 + db2') -> S3 (in place), partial of d eta
      float ln_mu, ln_rstd, ln_s1, ln_s2;
      {
        float z[16], tg[16];
        tmem_ld16(tmem + lane_addr + TM_S2 + c0, reinterpret_cast<uint32_t*>(z));
        {
          float kk[16];
          ld_row16(sbase + SM_TK, trow, 2 * cq, kk);
          ld_row16(sbase + SM_TV, trow, 2 * cq, tg);
#pragma unroll
          for (int f = 0; f < 16; ++f) tg[f] -= kk[f];  // target
        }
        tc_wait_ld();
        float a1 = 0.f, a2 = 0.f;
#pragma unroll
        for (int f = 0; f < 16; ++f) { z[f] += b2t[c0 + f]; a1 += z[f]; a2 = fmaf(z[f], z[f], a2); }
        xB[cq * 64 + trow] = make_float2(a1, a2);
        __syncthreads();
        a1 = 0.f; a2 = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float2 v = xB[q * 64 + trow]; a1 += v.x; a2 += v.y; }
        ln_mu = a1 * (1.f / 64.f);
        ln_rstd = rsqrtf(fmaxf(a2 * (1.f / 64.f) - ln_mu * ln_mu, 0.f) + 1e-8f);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int f = 0; f < 16; ++f) {
          z[f] = (z[f] - ln_mu) * ln_rstd;                                          // x_hat
          tg[f] = (fmaf(lnw[c0 + f], z[f], lnb[c0 + f]) - tg[f]) * lnw[c0 + f];      // gxh
          s1 += tg[f];
          s2 = fmaf(tg[f], z[f], s2);
        }
        *reinterpret_cast<float2*>(&xA[cq * 64 + trow]) = make_float2(s1, s2);
        __syncthreads();
        s1 = 0.f; s2 = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float4 v = xA[q * 64 + trow]; s1 += v.x; s2 += v.y; }
        ln_s1 = s1; ln_s2 = s2;
        const float neg_eta = etas[trow];
#pragma unroll
        for (int f = 0; f < 16; ++f) z[f] = (fmaf(64.f, tg[f], -s1) - z[f] * s2) * (ln_rstd * (1.f / 64.f));  // gradZ2
        st_row16(sbase + SM_TT1, trow, 2 * cq, z);
#pragma unroll
        for (int f = 0; f < 16; ++f) tg[f] = neg_eta * z[f];
        st_row16(sbase + SM_TT2, trow, 2 * cq, tg);
        tmem_ld16(tmem + lane_addr + TM_S3 + c0, reinterpret_cast<uint32_t*>(tg));  // acc5
        tc_wait_ld();
        float e = 0.f;
#pragma unroll
        for (int f = 0; f < 16; ++f) {
          const float a = tg[f] + db2c[c0 + f];
          e = fmaf(-z[f], a, e);
          tg[f] = neg_eta * a;
        }
        epart[cq * 64 + trow] = e;
        tmem_st16(tmem + lane_addr + TM_S3 + c0, reinterpret_cast<uint32_t*>(tg));
        tc_wait_st();
      }
      if (warp_u == 0 && elect_one()) bulk_wait_read<0>();  // X2 tile has been read out of smem: slot sC may be overwritten
      PHASE_SYNC();
      TICK(5);

      // ===== A5/A6 (two chunks of 32 tokens): pre = W2 . gradZ2^T -> S0, raw = CW1 . K^T -> S1 (N = 32);
      //       [H]: gradZ1, d gradZ1, DG1 -> sW1, G1eta -> sC, term2, d eta hidden-sums
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        if (warp_u == 0 && elect_one()) {
          tc_fence_after();
          mma_hid(tmem + TM_S0, tmem + TM_S0 + 32, sbase + SM_W2I, sbase + SM_TT1 + ch * 4096, false, 32, false);
          mma_hid(tmem + TM_S1, tmem + TM_S1 + 32, sbase + sA, sbase + SM_TK + ch * 4096, false, 32, false);
          tc_commit(mma_bar);
        }
        MMA_WAIT();
      TICK(6);
        {
          float pre[32], raw[32];
          tmem_ld32(tmem + lane_addr + TM_S0 + 32 * half, reinterpret_cast<uint32_t*>(pre));
          tmem_ld32(tmem + lane_addr + TM_S1 + 32 * half, reinterpret_cast<uint32_t*>(raw));
          tc_wait_ld();
          float ep[32];
          const f32x2 DB1 = pk2(db1r);
#pragma unroll
          for (int i = 0; i < 32; i += 2) {  // two tokens per instruction (FFMA2)
            const f32x2 g1 = bf16x2_to_f32x2(g1p[16 * ch + i / 2]), g2 = bf16x2_to_f32x2(g2p[16 * ch + i / 2]);
            const f32x2 net = *reinterpret_cast<const f32x2*>(&etas[32 * ch + i]);  // -eta of the two tokens
            const f32x2 pr = pk2(pre[i], pre[i + 1]);
            const f32x2 gz = mul2(pr, g1);                                  // gradZ1
            const f32x2 E = add2(pk2(raw[i], raw[i + 1]), DB1);
            const f32x2 d = mul2(net, E);                                   // d gradZ1
            up2(mul2(gz, E), ep[i], ep[i + 1]);
            g2p[16 * ch + i / 2] = pack_bf16(mul2(mul2(pr, d), g2));        // term2
            up2(mul2(d, g1), raw[i], raw[i + 1]);                           // DG1
            up2(mul2(net, gz), pre[i], pre[i + 1]);                         // G1eta
          }
          st_row32(sbase + sW1, j, 4 * ch, raw);
          st_row32(sbase + sC, j, 4 * ch, pre);
          warp_colsum<32>(ep, lane);
          esum8[((warp >> 1) * 64 + 32 * ch + lane) * 4 + 2 + (warp & 1)] = ep[0];  // partial of this warp's 32 hidden lanes
        }
        PHASE_SYNC();
      TICK(7);
      }
      // ===== A7 MMA: dK acc: S0 = G1eta . CW1 ; S3 += DG1 . W2
      if (warp_u == 0 && elect_one()) {
        tc_fence_after();
        mma_tok(tmem + TM_S0, sbase + sC, sbase + sA, false);
        mma_tok(tmem + TM_S3, sbase + sW1, sbase + SM_W2I, true);
        tc_commit(mma_bar);
      }
      MMA_WAIT();
      TICK(8);
      if (warp_u == 0 && elect_one()) {  // sA (CW1) and sC (G1eta) are free: reload the W1 image and the X2 tile
        bulk_wait<0>();
        mbar_expect_tx(bar_w1r, 32768);
        bulk_load_1d(smem + sA, img_at(cur), 32768, bar_w1r);
        mbar_expect_tx(bar_x2, 32768);
        bulk_load_1d(smem + sC, p.x2spill + (size_t)bh * kX2SpillBytes, 32768, bar_x2);
      }
      // ===== A8 [T] (all warps): stage 2 = backward through the fused LN + L2 gradient (appendix B), dZ2 -> TT0, dV,
      //       d eta, +dy (= -dtarget) folded into the dK accumulator S0, column sums for d b2 / d gamma / d beta
      {
        float z[16], go[16], dg[16];
        tmem_ld16(tmem + lane_addr + TM_S2 + c0, reinterpret_cast<uint32_t*>(z));
        tmem_ld16(tmem + lane_addr + TM_S3 + c0, reinterpret_cast<uint32_t*>(dg));
        {
          float kk[16];
          ld_row16(sbase + SM_TK, trow, 2 * cq, kk);
          ld_row16(sbase + SM_TV, trow, 2 * cq, go);
#pragma unroll
          for (int f = 0; f < 16; ++f) go[f] -= kk[f];  // target
        }
        tc_wait_ld();
        float sd = 0.f, sdx = 0.f;
#pragma unroll
        for (int f = 0; f < 16; ++f) {
          z[f] = (z[f] + b2t[c0 + f] - ln_mu) * ln_rstd;                 // x_hat
          go[f] = fmaf(lnw[c0 + f], z[f], lnb[c0 + f]) - go[f];           // grad_output
          sd += dg[f];
          sdx = fmaf(dg[f], z[f], sdx);
        }
        xB[cq * 64 + trow] = make_float2(sd, sdx);
        __syncthreads();
        sd = 0.f; sdx = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float2 v = xB[q * 64 + trow]; sd += v.x; sdx += v.y; }
        float sds = 0.f, sdxh = 0.f;
        float dy[16], cg[16];
#pragma unroll
        for (int f = 0; f < 16; ++f) {
          const float gam = lnw[c0 + f];
          const float gxh = go[f] * gam;
          const float gz2 = (fmaf(64.f, gxh, -ln_s1) - z[f] * ln_s2) * (ln_rstd * (1.f / 64.f));
          const float dgxh = ln_rstd * (dg[f] - (1.f / 64.f) * (sd + z[f] * sdx));
          dy[f] = gam * dgxh;
          cg[f] = fmaf(go[f], dgxh, dy[f] * z[f]);                                   // d gamma contribution
          const float dxh = fmaf(dy[f], gam, -(ln_rstd * (1.f / 64.f)) * fmaf(gxh, sdx, dg[f] * ln_s2));
          sds += (-dxh * z[f] - dg[f] * gz2) * ln_rstd;
          sdxh += dxh;
          dg[f] = dxh;                                                               // keep d_xhat
        }
        *reinterpret_cast<float2*>(&xA[cq * 64 + trow]) = make_float2(sds, sdxh);  // .z/.w hold the d eta partials
        __syncthreads();
        sds = 0.f; sdxh = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float4 v = xA[q * 64 + trow]; sds += v.x; sdxh += v.y; }
#pragma unroll
        for (int f = 0; f < 16; ++f) dg[f] = fmaf(dg[f], ln_rstd, (1.f / 64.f) * (z[f] * sds - sdxh * ln_rstd));  // dZ2
        st_row16(sbase + SM_TT0, trow, 2 * cq, dg);
        {  // dV = dtarget = -dy
          float nd[16];
#pragma unroll
          for (int f = 0; f < 16; ++f) nd[f] = -dy[f];
          st_global16(p.dXV + (row_bh + (size_t)t * CS + trow) * F + c0, nd);
        }
        {  // fold -dtarget (= +dy) into the dK accumulator S0 (this thread's lane copy, its own 16 columns)
          float a[16];
          tmem_ld16(tmem + lane_addr + TM_S0 + c0, reinterpret_cast<uint32_t*>(a));
          tc_wait_ld();
#pragma unroll
          for (int f = 0; f < 16; ++f) a[f] += dy[f];
          tmem_st16(tmem + lane_addr + TM_S0 + c0, reinterpret_cast<uint32_t*>(a));
          tc_wait_st();
        }
        if (cq == 0) {  // d eta of step t
          float es = 0.f;
#pragma unroll
          for (int w = 0; w < 8; ++w) es += esum8[((w >> 1) * 64 + trow) * 4 + 2 + (w & 1)];  // fixed order
          const float e = epart[trow] + epart[64 + trow] + epart[128 + trow] + epart[192 + trow] - es;
          p.dEta[row_bh + (size_t)t * CS + trow] = __float2bfloat16(e);
        }
        // column sums over this warp's 32 token rows (then shared atomics across the two row halves)
        warp_colsum16(dg, lane);
        warp_colsum16(cg, lane);
        warp_colsum16(dy, lane);
        if ((lane & 1) == 0) {
          const int f = c0 + (lane >> 1);
          const bool hi = (warp & 1) != 0;  // token rows 32-63: the other accumulator set (one writer per word)
          atomicAdd(&(hi ? db2h : db2c)[f], dg[0]);  // fire-and-forget shared-memory adds; each word has ONE writer per step
          atomicAdd(&(hi ? dgam2 : dgam)[f], cg[0]);
          atomicAdd(&(hi ? dbet2 : dbet)[f], dy[0]);
        }
      }
      PHASE_SYNC();
      TICK(9);
      // ===== A9 MMA: dX2^T = W2 . dZ2^T + CW2 . (-eta gradZ2)^T -> (S1,S2)   (waited)
      //       then, not waited here: dW2 += DG1^T gradZ2 + X2^T dZ2 -- their completion (bar_aux) frees the DG1 and X2
      //       slots early so that next iteration's tiles stream in under A10/A11
      mbar_wait(bar_x2, ph_x2); ph_x2 ^= 1;
      if (warp_u == 0 && elect_one()) {
        tc_fence_after();
        mma_hid(tmem + TM_S1, tmem + TM_S2, sbase + SM_W2I, sbase + SM_TT0, false, 64, false);
        mma_hid(tmem + TM_S1, tmem + TM_S2, sbase + sB, sbase + SM_TT2, false, 64, true);
        tc_commit(mma_bar);
        mma_hid(tmem + TM_DW2, tmem + TM_DW2 + 64, sbase + sW1, sbase + SM_TT1, true, 64, true);
        mma_hid(tmem + TM_DW2, tmem + TM_DW2 + 64, sbase + sC, sbase + SM_TT0, true, 64, true);
        tc_commit(bar_aux);
      }
      MMA_WAIT();
      TICK(10);
      if (warp_u == 0 && (t > p.t_lo) && elect_one()) {  // the W2 image buffer is free now: fetch the next one
        mbar_expect_tx(bar_w2, 32768);
        bulk_load_1d(smem + SM_W2I, img_at(nxt) + kImageW2, 32768, bar_w2);
      }
      // ===== A10 [H]: dZ1 = dX2 * gelu'(Z1) + term2 -> sB ; d b1 += sum dZ1
      {
        const uint32_t src = tmem + lane_addr + (half ? TM_S2 : TM_S1);
        f32x2 acc2 = pk2(0.f);  // even / odd tokens
        float v[2][32];
        tmem_ld32(src, reinterpret_cast<uint32_t*>(v[0]));
        tmem_ld32(src + 32, reinterpret_cast<uint32_t*>(v[1]));
        tc_wait_ld();
#pragma unroll
        for (int c = 0; c < 2; ++c) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const f32x2 r = fma2(pk2(v[c][i], v[c][i + 1]), bf16x2_to_f32x2(g1p[16 * c + i / 2]), bf16x2_to_f32x2(g2p[16 * c + i / 2]));
            up2(r, v[c][i], v[c][i + 1]);
            acc2 = add2(acc2, r);
          }
          st_row32(sbase + sB, j, 4 * c, v[c]);
        }
        db1r += lo2(acc2) + hi2(acc2);
      }
      mbar_wait(bar_w1r, ph_w1r); ph_w1r ^= 1;
      mbar_wait(bar_aux, ph_aux); ph_aux ^= 1;   // DG1 (sW1) and X2 (sC) are no longer read by any MMA
      if (warp_u == 0 && (t > p.t_lo) && elect_one()) {
        mbar_expect_tx(bar_w1, 32768);
        bulk_load_1d(smem + sC, img_at(nxt), 32768, bar_w1);
        load_xb(t - 1, sW1);
      }
      PHASE_SYNC();
      TICK(11);
      // ===== A11 MMA: dK: S0 += dZ1 . W1 ; dW1^T += dZ1^T K
      if (warp_u == 0 && elect_one()) {
        tc_fence_after();
        mma_tok(tmem + TM_S0, sbase + sB, sbase + sA, true);
        mma_hid(tmem + TM_DW1, tmem + TM_DW1 + 64, sbase + sB, sbase + SM_TK, true, 64, true);
        tc_commit(mma_bar);
      }
      MMA_WAIT();
      TICK(12);
      // ===== A12 [T]: dK -> global
      {
        float a[16];
        tmem_ld16(tmem + lane_addr + TM_S0 + c0, reinterpret_cast<uint32_t*>(a));
        tc_wait_ld();
        st_global16(p.dXK + (row_bh + (size_t)t * CS + trow) * F + c0, a);
      }
      tc_fence_before();
      __syncthreads();
      TICK(13);
    }

    // persistent mode: step t was the last access to its unit's recompute buffers -> the trajectory kernel that refills this
    // ring slot (unit u + kRingSlots) may start (every bulk load of the unit has completed and was consumed above)
    if (p.done != nullptr && t % p.G == 0 && tid == 0) release_flag<kSet>(p.done + (size_t)unit_of_group(t / p.G, p.K) * gridDim.x + bh);
    // next iteration's remaining loads (buffers last used by the A11 batch): K/V tiles, Q tile, dZbar1^T -> sA, dZbar2 -> TT0
    const bool more = t > p.t_lo;
    if (warp_u == 0 && (more) && elect_one()) {
      const int tn = t - 1;
      mbar_expect_tx(bar_kv, 16384);
      tma_load_2d(smem + SM_TK, &tmK, 0, (int)(row_bh + (size_t)tn * CS), bar_kv);
      tma_load_2d(smem + SM_TV, &tmV, 0, (int)(row_bh + (size_t)tn * CS), bar_kv);
      load_q_rest(tn, sA);
    }
    // rotate slot roles: the next W1 image was fetched into sC
    {
      const uint32_t n0 = sC, n1 = sW1, n2 = sA, n3 = sB;
      sW1 = n0; sA = n1; sB = n2; sC = n3;
    }
    // advance the step pointers: cur <- step t - 1, nxt <- step t - 2
    cur = nxt;
    tcur = t - 1;
    if (t - 1 > p.t_lo) step_back(nxt);
  }

  TICK(15);  // (loop tail)
  // ---- epilogue: carried gradient -> scratch (or final outputs), LN parameter gradients
  tc_fence_after();
  {
    const bool fin = (p.t_lo == 0);
    float v[32];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      tmem_ld32(tmem + lane_addr + TM_DW1 + 64 * half + 32 * c, reinterpret_cast<uint32_t*>(v));
      tc_wait_ld();
      if (fin) {
#pragma unroll
        for (int i = 0; i < 32; ++i) p.dW1[((size_t)bh * F + 32 * c + i) * HID + j] = v[i];  // [f][j] layout
      } else {
        float4* d1 = reinterpret_cast<float4*>(p.dW1s + ((size_t)bh * HID + j) * F + 32 * c);
#pragma unroll
        for (int i = 0; i < 8; ++i) d1[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      tmem_ld32(tmem + lane_addr + TM_DW2 + 64 * half + 32 * c, reinterpret_cast<uint32_t*>(v));
      tc_wait_ld();
      float4* dst = reinterpret_cast<float4*>((fin ? p.dW2 : p.dW2s) + ((size_t)bh * HID + j) * F + 32 * c);
#pragma unroll
      for (int i = 0; i < 8; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }
    (fin ? p.db1 : p.db1s)[(size_t)bh * HID + j] = db1r;
    if (tid < 64) (fin ? p.db2 : p.db2s)[(size_t)bh * 64 + tid] = db2c[tid] + db2h[tid];
    if (tid < 64) {  // launches of one sequence are stream-ordered and nobody else writes these words: plain accumulate
      p.dlnw[(size_t)bh * 64 + tid] += dgam[tid] + dgam2[tid];
      p.dlnb[(size_t)bh * 64 + tid] += dbet[tid] + dbet2[tid];
    }
  }
  TICK(16);  // epilogue stores
  if (p.t_lo / p.G == p.dbg_group) TICK_DUMP(22, p.dbg);
#ifdef TTT_PHASE_TIMING
  if (p.dbg && tid == 0 && blockIdx.x < 64) {  // per-block total cycles + SM id (placement effects)
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    p.dbg[128 + blockIdx.x] = (unsigned)(clock64() - tick_t0_64);
    p.dbg[192 + blockIdx.x] = smid;
    unsigned long long g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    const int gi = p.t_lo / p.G;  // block start / end wall time (ns, low 32 bits), one record per group (up to 27)
    if (gi < 27) {
      p.dbg[512 + gi * 128 + blockIdx.x] = (unsigned)tick_g0;
      p.dbg[512 + gi * 128 + 64 + blockIdx.x] = (unsigned)g1;
    }
  }
#endif
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

// Upstream gradient of the FINAL state (sequence-sharded chain: the next shard's d/dW_init) -> carried-gradient scratch in
// the kernel's layout (dW1 transposed to [hidden][F]); one block per sequence.
__global__ void seed_state_grad_kernel(const float* __restrict__ dW1u, const float* __restrict__ db1u,
                                       const float* __restrict__ dW2u, const float* __restrict__ db2u, float* dW1s,
                                       float* dW2s, float* db1s, float* db2s) {
  const size_t bh = blockIdx.x;
  __shared__ float tile[64][65];
  for (int jb = 0; jb < HID; jb += 64) {  // dW1u [F][HID] -> dW1s [HID][F]
    for (int i = threadIdx.x; i < 64 * 64; i += blockDim.x) tile[i >> 6][i & 63] = dW1u[(bh * F + (i >> 6)) * HID + jb + (i & 63)];
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * 64; i += blockDim.x) dW1s[(bh * HID + jb + (i >> 6)) * F + (i & 63)] = tile[i & 63][i >> 6];
    __syncthreads();
  }
  for (int i = threadIdx.x; i < HID * F; i += blockDim.x) dW2s[bh * HID * F + i] = dW2u[bh * HID * F + i];
  for (int i = threadIdx.x; i < HID; i += blockDim.x) db1s[bh * HID + i] = db1u[bh * HID + i];
  for (int i = threadIdx.x; i < F; i += blockDim.x) db2s[bh * F + i] = db2u[bh * F + i];
}

}  // namespace bwd

// ------------------------------------------------------------------------------------------------ host
// Recompute state is kept in a ring of kRingSlots buffers (recompute_ring.cuh) so that the trajectory / Q-side kernels of later units run ahead of the
// sequential K-side kernel (three streams).  A unit = one checkpoint group, processed last group first.
//
// Persistent mode (default when 2 * B*H + 16 <= SM count): ONE K-side launch walks all units; the recompute kernels run
// beside it on the other SMs and the three kernels hand-shake through device-side counters (BwdParams::ready / done)
// instead of host events -- no per-group launch gap, no carried-gradient round trip through global memory, no cold
// instruction fetch per group (measured round 1: ~54 us per group of 16 steps, 19 % of the backward).  All recompute
// launches are enqueued up front: a trajectory kernel whose ring slot is still in use spins (bounded, traps on timeout)
// until the K-side CTA of its sequence releases the slot.  The SM-count condition keeps SMs free for the Q-side kernel
// while B*H K-side CTAs and up to B*H waiting trajectory CTAs are resident (one CTA of any of the three kernels fills an
// SM); above it the launches are ordered per unit with events as in round 1 (TTT_B200_PERSISTENT=0 forces that mode).
size_t mlp_backward_workspace_bytes(int B, int H, int G) { return carve_mlp_workspace(nullptr, (size_t)B * H, G, nullptr); }

cudaError_t launch_mlp_backward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                const float* ln_b, const float* W1c, const float* b1c, const float* W2c,
                                const float* b2c, const void* dOut, float* dlnw, float* dlnb, float* dW1, float* db1,
                                float* dW2, float* db2, void* dEta, void* dXQ, void* dXK, void* dXV, void* workspace,
                                size_t workspace_bytes, int B, int H, int NC, int G, cudaStream_t stream,
                                const float* dW1_last, const float* db1_last, const float* dW2_last,
                                const float* db2_last) {
  if (B <= 0 || H <= 0 || NC <= 0 || G <= 0) { g_where = "bad sizes"; return cudaErrorInvalidValue; }
  if (workspace_bytes < mlp_backward_workspace_bytes(B, H, G)) { g_where = "workspace"; return cudaErrorInvalidValue; }
  const size_t bh = (size_t)B * H;
  const int K = (NC + G - 1) / G;  // units = checkpoint groups
  if (K > kMaxUnits) { g_where = "too many checkpoint groups"; return cudaErrorInvalidValue; }
  MlpWorkspace ws;
  carve_mlp_workspace(workspace, bh, G, &ws);

  CUtensorMap tq, tk, tv, tdo;
  const uint64_t rows = (uint64_t)bh * NC * 64;
  if (rows > 0x7FFFFFFFull) { g_where = "too many rows"; return cudaErrorInvalidValue; }
  if (make_token_tmap(&tq, XQ, rows) || make_token_tmap(&tk, XK, rows) || make_token_tmap(&tv, XV, rows) ||
      make_token_tmap(&tdo, dOut, rows)) return cudaErrorInvalidValue;  // g_where set by make_token_tmap
  std::lock_guard<std::mutex> enqueue_lock(device_enqueue_mutex());
  static bool attr_done_dev[64] = {};  // function attributes (and side streams) are per device
  static int sm_count_dev[64] = {};
  bool& attr_done = *device_once(attr_done_dev);
  int dev = 0;
  TB_TRY(cudaGetDevice(&dev), "cudaGetDevice");
  if (!attr_done) {
    TB_TRY(cudaFuncSetAttribute(bwd::ttt_mlp_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd::SM_TOTAL), "smem attr");
    TB_TRY(cudaDeviceGetAttribute(&sm_count_dev[dev & 63], cudaDevAttrMultiProcessorCount, dev), "SM count");
    attr_done = true;
  }
  TB_TRY(cudaMemsetAsync(dlnw, 0, bh * 64 * sizeof(float), stream), "memset dlnw");
  TB_TRY(cudaMemsetAsync(dlnb, 0, bh * 64 * sizeof(float), stream), "memset dlnb");

  // three streams per device (created once): T = trajectory, Q = Q-side kernel, main = sequential K-side kernel
  struct Side {
    cudaStream_t sT = nullptr, sQ = nullptr;
    cudaEvent_t fork = nullptr, joinT = nullptr, joinQ = nullptr, evT[kRingSlots] = {}, evQ[kRingSlots] = {}, evR[kRingSlots] = {};
  };
  static Side sides[64];
  Side& sd = sides[dev & 63];
  if (!sd.sT) {
    int prio_lo = 0, prio_hi = 0;  // recompute work must never delay the CTAs of the sequential kernel: lowest priority
    TB_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi), "priority range");
    TB_TRY(cudaStreamCreateWithPriority(&sd.sT, cudaStreamNonBlocking, prio_lo), "side stream");
    TB_TRY(cudaStreamCreateWithPriority(&sd.sQ, cudaStreamNonBlocking, prio_lo), "side stream");
    TB_TRY(cudaEventCreateWithFlags(&sd.fork, cudaEventDisableTiming), "event");
    TB_TRY(cudaEventCreateWithFlags(&sd.joinT, cudaEventDisableTiming), "event");
    TB_TRY(cudaEventCreateWithFlags(&sd.joinQ, cudaEventDisableTiming), "event");
    for (int i = 0; i < kRingSlots; ++i) {
      TB_TRY(cudaEventCreateWithFlags(&sd.evT[i], cudaEventDisableTiming), "event");
      TB_TRY(cudaEventCreateWithFlags(&sd.evQ[i], cudaEventDisableTiming), "event");
      TB_TRY(cudaEventCreateWithFlags(&sd.evR[i], cudaEventDisableTiming), "event");
    }
  }
  static const int dbg_group_env = [] { const char* v = getenv("TTT_DBG_GROUP"); return v ? atoi(v) : 0; }();
  static const int persistent_env = [] { const char* v = getenv("TTT_B200_PERSISTENT"); return v ? atoi(v) : 1; }();
  const bool persistent = persistent_env != 0 && 2 * (int)bh + 16 <= sm_count_dev[dev & 63];
  const bool seeded = dW1_last != nullptr;
  if (seeded) {  // carried gradient starts from the upstream d/dW_last instead of zero
    bwd::seed_state_grad_kernel<<<(unsigned)bh, 256, 0, stream>>>(dW1_last, db1_last, dW2_last, db2_last, ws.dW1s, ws.dW2s, ws.db1s,
                                                                   ws.db2s);
    TB_TRY(cudaGetLastError(), "seed launch");
  }
  if (persistent) {
    TB_TRY(cudaMemsetAsync(ws.ready, 0, bh * (size_t)K * sizeof(unsigned), stream), "memset ready flags");
    TB_TRY(cudaMemsetAsync(ws.done, 0, bh * (size_t)K * sizeof(unsigned), stream), "memset done flags");
  }
  // unit u: trajectory (images of W_{t0} .. W_{t1}) on stream T, then the Q-side kernel (steps t0 .. t1-1) on stream Q
  auto recompute = [&](int u) -> cudaError_t {
    const int r = ring_slot(u), g = unit_of_group(u, K);
    const int t0 = group_begin(g, G), t1 = group_end(g, G, NC);
    const unsigned* wait_done = (persistent && u >= kRingSlots) ? ws.done + (size_t)(u - kRingSlots) * bh : nullptr;
    cudaError_t e = launch_mlp_trajectory_compact(XK, XV, last_eta, ln_w, ln_b, W1c, b1c, W2c, b2c, B, H, NC, K, G, t0, t1,
                                                  ws.ring[r], sd.sT, wait_done);
    if (e != cudaSuccess) return e;
    if ((e = cudaEventRecord(sd.evT[r], sd.sT)) != cudaSuccess) return e;
    if ((e = cudaStreamWaitEvent(sd.sQ, sd.evT[r], 0)) != cudaSuccess) return e;
    e = launch_mlp_backward_q(tq, tdo, ln_w, ln_b, ws.ring[r], dXQ, (int)bh, H, NC, G, t0, t1 - t0, sd.sQ,
                              persistent ? ws.ready + (size_t)u * bh : nullptr);
    if (e != cudaSuccess) return e;
    return cudaEventRecord(sd.evQ[r], sd.sQ);
  };
  bwd::BwdParams p{};
  p.last_eta = reinterpret_cast<const __nv_bfloat16*>(last_eta);
  p.ln_w = ln_w; p.ln_b = ln_b;
  for (int i = 0; i < kRingSlots; ++i) p.ring[i] = ws.ring[i];
  p.dW1s = ws.dW1s; p.dW2s = ws.dW2s; p.db1s = ws.db1s; p.db2s = ws.db2s;
  p.x2spill = ws.x2spill;
  p.G = G; p.K = K;
  p.dXQ = reinterpret_cast<__nv_bfloat16*>(dXQ); p.dXK = reinterpret_cast<__nv_bfloat16*>(dXK);
  p.dXV = reinterpret_cast<__nv_bfloat16*>(dXV); p.dEta = reinterpret_cast<__nv_bfloat16*>(dEta);
  p.dlnw = dlnw; p.dlnb = dlnb;
  p.dW1 = dW1; p.db1 = db1; p.dW2 = dW2; p.db2 = db2;
  p.H = H; p.NC = NC; p.img_slots = G + 1;
  p.dbg_group = dbg_group_env;
  p.dbg = g_timing_buf;  // observers: the launch whose t_lo / G equals TTT_DBG_GROUP; per-launch stamps are kept

  TB_TRY(cudaEventRecord(sd.fork, stream), "fork record");
  TB_TRY(cudaStreamWaitEvent(sd.sT, sd.fork, 0), "fork wait");
  TB_TRY(cudaStreamWaitEvent(sd.sQ, sd.fork, 0), "fork wait");
  for (int i = 0; i < kRingSlots && i < K; ++i) TB_TRY(recompute(i), "trajectory / Q launch");

  if (persistent) {
    p.t_hi = NC - 1; p.t_lo = 0;
    p.first = seeded ? 0 : 1;
    p.ready = ws.ready; p.done = ws.done;
    bwd::ttt_mlp_bwd_kernel<<<(unsigned)bh, bwd::NT, bwd::SM_TOTAL, stream>>>(tq, tk, tv, p);
    TB_TRY(cudaGetLastError(), "reverse launch (persistent)");
    for (int u = kRingSlots; u < K; ++u) TB_TRY(recompute(u), "trajectory / Q launch");  // each waits on-device for its ring slot
  } else {
    for (int u = 0; u < K; ++u) {
      const int r = ring_slot(u), g = unit_of_group(u, K);
      TB_TRY(cudaStreamWaitEvent(stream, sd.evQ[r], 0), "wait Q-side");
      p.t_hi = group_end(g, G, NC) - 1;
      p.t_lo = group_begin(g, G);
      p.first = (u == 0 && !seeded) ? 1 : 0;
      bwd::ttt_mlp_bwd_kernel<<<(unsigned)bh, bwd::NT, bwd::SM_TOTAL, stream>>>(tq, tk, tv, p);
      TB_TRY(cudaGetLastError(), "reverse launch");
      if (u + kRingSlots < K) {  // ring buffer r is free again once this launch is done: recompute unit u + kRingSlots into it
        TB_TRY(cudaEventRecord(sd.evR[r], stream), "record reverse");
        TB_TRY(cudaStreamWaitEvent(sd.sT, sd.evR[r], 0), "wait reverse");
        TB_TRY(recompute(u + kRingSlots), "trajectory / Q launch");
      }
    }
  }
  // join: later work on `stream` (and the next call, which reuses the side streams and this workspace) is ordered after
  // everything enqueued on the side streams
  TB_TRY(cudaEventRecord(sd.joinT, sd.sT), "join record");
  TB_TRY(cudaEventRecord(sd.joinQ, sd.sQ), "join record");
  TB_TRY(cudaStreamWaitEvent(stream, sd.joinT, 0), "join wait");
  TB_TRY(cudaStreamWaitEvent(stream, sd.joinQ, 0), "join wait");
  return cudaSuccess;
}

}  // namespace tb
