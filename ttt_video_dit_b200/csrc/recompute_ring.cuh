// Recompute buffers of the backward passes and their hand-off protocol: the one place that knows the workspace layout.
//
// TTT-MLP (DESIGN.md section 4): the checkpoint groups are processed last group first; group g (steps
// [g*G, min((g+1)*G, NC))) is recompute unit u = K-1-g and lives in ring slot u % kRingSlots.  Per slot and sequence the
// trajectory kernel (ttt_mlp_traj.cu) writes the state images of the G + 1 states the group passes through, the Q-side
// kernel (ttt_mlp_bwd_q.cu) reads them and writes one factor record per step, and the K-side kernel (ttt_mlp_bwd.cu) reads
// both.  In persistent K-side mode the three kernels hand-shake through the ready / done flags below.
//
// TTT-Linear (DESIGN.md section 4b): the trajectory-mode forward (ttt_linear_fwd.cu) writes the state image of every step
// of a recompute window for a PAIR of sequences (the two W1^T stacked on the 128 TMEM lanes), the reverse kernel
// (ttt_linear_bwd.cu) reads its own half.  One or two window buffers.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

namespace tb {

// ------------------------------------------------------------------------------------------------ TTT-MLP records
constexpr int kRingSlots = 3;     // recompute units in flight
constexpr int kMaxUnits = 4096;   // checkpoint groups per call (ready / done flags per sequence)

// state image: bf16 operand tiles ([256][64], SW128 rows) of the state entering a step
constexpr size_t kImageBytes = 65536;
constexpr size_t kImageW1T = 0, kImageW2 = 32768;
constexpr int kImageB1Floats = 256, kImageB2Floats = 64;  // fp32 b1 / b2 of the same state
// Q-side factor record of a step: bf16 tiles Xbar2^T [256][64], dZbar1^T [256][64], dZbar2 [64][64]
constexpr size_t kFactorBytes = 73728;
constexpr size_t kFactorXbar2T = 0, kFactorDZbar1T = 32768, kFactorDZbar2 = 65536;
constexpr int kFactorB1Floats = 256;  // sum over tokens of dZbar1
constexpr int kFactorVecFloats = 192, kFactorDb2 = 0, kFactorDgamma = 64, kFactorDbeta = 128;  // {d b2, d gamma, d beta}
constexpr size_t kX2SpillBytes = 32768;  // K-side X2 tile [256][64] bf16, per sequence

// one ring slot; `img_slots` = G + 1 image records and G factor records per sequence
struct MlpSlot {
  uint8_t* img;
  float *b1img, *b2img;
  uint8_t* qt;
  float *qb1, *qb2;
  __host__ __device__ __forceinline__ uint8_t* image(size_t bh, int img_slots, int l) const { return img + (bh * img_slots + l) * kImageBytes; }
  __host__ __device__ __forceinline__ float* image_b1(size_t bh, int img_slots, int l) const { return b1img + (bh * img_slots + l) * kImageB1Floats; }
  __host__ __device__ __forceinline__ float* image_b2(size_t bh, int img_slots, int l) const { return b2img + (bh * img_slots + l) * kImageB2Floats; }
  __host__ __device__ __forceinline__ uint8_t* factors(size_t bh, int G, int l) const { return qt + (bh * G + l) * kFactorBytes; }
  __host__ __device__ __forceinline__ float* factor_b1(size_t bh, int G, int l) const { return qb1 + (bh * G + l) * kFactorB1Floats; }
  __host__ __device__ __forceinline__ float* factor_vec(size_t bh, int G, int l) const { return qb2 + (bh * G + l) * kFactorVecFloats; }
};

struct MlpWorkspace {
  MlpSlot ring[kRingSlots];
  uint8_t* x2spill;                  // [BH] x kX2SpillBytes
  float *dW1s, *dW2s, *db1s, *db2s;  // carried state gradient, fp32: [BH][256][64] x2, [BH][256], [BH][64]
  unsigned *ready, *done;            // persistent mode: [kMaxUnits + 1][BH] each
};

// Bump allocator over a workspace; with a null base it only counts.
class Carve {
 public:
  explicit Carve(void* base) : p_(reinterpret_cast<uintptr_t>(base)) {}
  template <class T> T* take(size_t bytes) { T* r = reinterpret_cast<T*>(p_ + n_); n_ += bytes; return r; }
  size_t bytes() const { return n_; }
 private:
  uintptr_t p_;
  size_t n_ = 0;
};

// Lays the TTT-MLP workspace out from `base` rounded up to 1024 B and returns the bytes it needs (1024 of slack for
// the rounding included).  base == nullptr: the size only.
inline size_t carve_mlp_workspace(void* base, size_t BH, int G, MlpWorkspace* ws) {
  const size_t slots = (size_t)G + 1;
  Carve c(base ? reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(base) + 1023) & ~(uintptr_t)1023) : nullptr);
  MlpWorkspace w;
  for (MlpSlot& s : w.ring) s.img = c.take<uint8_t>(BH * slots * kImageBytes);
  w.x2spill = c.take<uint8_t>(BH * kX2SpillBytes);
  w.dW1s = c.take<float>(BH * 256 * 64 * sizeof(float));
  w.dW2s = c.take<float>(BH * 256 * 64 * sizeof(float));
  for (MlpSlot& s : w.ring) s.b1img = c.take<float>(BH * slots * kImageB1Floats * sizeof(float));
  for (MlpSlot& s : w.ring) s.b2img = c.take<float>(BH * slots * kImageB2Floats * sizeof(float));
  w.db1s = c.take<float>(BH * 256 * sizeof(float));
  w.db2s = c.take<float>(BH * 64 * sizeof(float));
  for (MlpSlot& s : w.ring) s.qt = c.take<uint8_t>(BH * G * kFactorBytes);
  for (MlpSlot& s : w.ring) s.qb1 = c.take<float>(BH * G * kFactorB1Floats * sizeof(float));
  for (MlpSlot& s : w.ring) s.qb2 = c.take<float>(BH * G * kFactorVecFloats * sizeof(float));
  w.ready = c.take<unsigned>(BH * (kMaxUnits + 1) * sizeof(unsigned));
  w.done = c.take<unsigned>(BH * (kMaxUnits + 1) * sizeof(unsigned));
  if (ws) *ws = w;
  return c.bytes() + 1024;
}

// ------------------------------------------------------------------------------------------------ units and groups
__host__ __device__ __forceinline__ int unit_of_group(int g, int K) { return K - 1 - g; }  // its own inverse
__host__ __device__ __forceinline__ int ring_slot(int u) { return u % kRingSlots; }
__host__ __device__ __forceinline__ int group_begin(int g, int G) { return g * G; }
__host__ __device__ __forceinline__ int group_end(int g, int G, int NC) { return min(NC, (g + 1) * G); }

// ------------------------------------------------------------------------------------------------ flags
// Bounded spin until *flag >= want, written by another kernel (acquire at gpu scope).  A protocol bug must surface as a
// launch failure (trap), never as a hung GPU.  The data behind the flag may be read by bulk / TMA loads (async proxy).
template <unsigned kSleepNs>
__device__ __forceinline__ void wait_flag(const unsigned* flag, unsigned want) {
  const long long t0 = clock64();
  for (;;) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if (v >= want) break;
    __nanosleep(kSleepNs);
    if (clock64() - t0 > 20000000000LL) {
      printf("ttt_b200: device-side flag wait timed out (block %d thread %d, have %u want %u)\n", (int)blockIdx.x, (int)threadIdx.x, v, want);
      __trap();
    }
  }
  asm volatile("fence.proxy.async;" ::: "memory");
}

// Publishes every global store this thread has ordered before the call (the CTA's, behind a __syncthreads) at gpu scope:
// kSet stores 1 (a flag with one writer), kCount adds 1 (a counter that several CTAs bump).
enum FlagRelease { kSet, kCount };
template <FlagRelease kOp>
__device__ __forceinline__ void release_flag(unsigned* flag) {
  __threadfence();
  if (kOp == kCount) asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(flag), "r"(1u) : "memory");
  else               asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(1u) : "memory");
}

// ------------------------------------------------------------------------------------------------ TTT-Linear records
// state image of a sequence pair: W1^T of sequence 2p at +0 and of 2p+1 at +8192 ([64][64] bf16 each, SW128 rows); fp32
// b1 of both, 64 floats each
constexpr size_t kLinImageBytes = 16384, kLinSeqImageBytes = 8192;
constexpr int kLinImageB1Floats = 128, kLinSeqB1Floats = 64;
constexpr int kLinMaxBuffers = 2;  // window buffers: the reverse pass over window w overlaps the recompute of w - 1

// one window buffer; `img_slots` = window steps + 1 records per pair
struct LinearImages {
  uint8_t* img;
  float* b1img;
  __host__ __device__ __forceinline__ uint8_t* image(size_t pair, int img_slots, int l) const { return img + (pair * img_slots + l) * kLinImageBytes; }
  __host__ __device__ __forceinline__ float* image_b1(size_t pair, int img_slots, int l) const { return b1img + (pair * img_slots + l) * kLinImageB1Floats; }
};

// Lays out `nbuf` window buffers of `img_slots` records per pair from `base` and returns the bytes they need (1024 B of
// slack included).  base == nullptr: the size only.
inline size_t carve_linear_workspace(void* base, size_t pairs, size_t img_slots, int nbuf, LinearImages* bufs) {
  if (nbuf < 1 || nbuf > kLinMaxBuffers) return 0;
  Carve c(base);
  LinearImages b[kLinMaxBuffers] = {};
  for (int i = 0; i < nbuf; ++i) b[i].img = c.take<uint8_t>(pairs * img_slots * kLinImageBytes);
  for (int i = 0; i < nbuf; ++i) b[i].b1img = c.take<float>(pairs * img_slots * kLinImageB1Floats * sizeof(float));
  if (bufs) for (int i = 0; i < nbuf; ++i) bufs[i] = b[i];
  return c.bytes() + 1024;
}

}  // namespace tb
