// Internal (non-ABI) declarations shared by the .cu files of libttt_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <mutex>
#include <stdint.h>

namespace tb {

// last failing step inside a multi-launch entry point (read by capi.cu for the error message)
extern thread_local const char* g_where;
extern unsigned* g_timing_buf;  // device buffer [2][64] for phase timing (debug builds), may be null
// per-device "done once" flag for launch-site initialisation: cudaFuncSetAttribute and streams / events belong to one device
inline bool* device_once(bool (&flags)[64]) {
  int d = 0;
  cudaGetDevice(&d);
  return &flags[d & 63];
}
// The backward orchestrators share per-device side streams and events; two host threads enqueueing on the same device are
// serialised for the duration of the (asynchronous) enqueue.  Different devices never contend.
inline std::mutex& device_enqueue_mutex() {
  static std::mutex mu[64];
  int d = 0;
  cudaGetDevice(&d);
  return mu[d & 63];
}

#define TB_TRY(call, what)                 \
  do {                                     \
    cudaError_t e__ = (call);              \
    if (e__ != cudaSuccess) {              \
      ::tb::g_where = (what);              \
      return e__;                          \
    }                                      \
  } while (0)

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_token_tmap(CUtensorMap* tm, const void* base, uint64_t rows);
int make_token_tmap_box(CUtensorMap* tm, const void* base, uint64_t rows, uint32_t box_rows);

cudaError_t launch_mlp_forward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                               const float* ln_b, const float* W1, const float* b1, const float* W2, const float* b2,
                               float* W1c, float* b1c, float* W2c, float* b2c, float* W1o, float* b1o, float* W2o,
                               float* b2o, void* Out, int B, int H, int NC, int ckpt_group, cudaStream_t stream);

cudaError_t launch_umma_selftest(int mode, const void* A, const void* Bm, float* D, int N, int K, cudaStream_t stream);

}  // namespace tb

namespace tb {
struct MlpSlot;  // recompute_ring.cuh
bool mlp_operands_bf16();  // TTT_B200_OPERANDS=bf16: bf16 instead of fp16 operand tiles in the forward-type kernels (A/B)
cudaError_t launch_mlp_trajectory_compact(const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                          const float* ln_b, const float* W1c, const float* b1c, const float* W2c,
                                          const float* b2c, int B, int H, int NC, int K, int G, int t0, int t_end,
                                          const MlpSlot& slot, cudaStream_t stream, const unsigned* wait_done = nullptr);
size_t mlp_backward_workspace_bytes(int B, int H, int G);
cudaError_t launch_mlp_backward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                const float* ln_b, const float* W1c, const float* b1c, const float* W2c,
                                const float* b2c, const void* dOut, float* dlnw, float* dlnb, float* dW1, float* db1,
                                float* dW2, float* db2, void* dEta, void* dXQ, void* dXK, void* dXV, void* workspace,
                                size_t workspace_bytes, int B, int H, int NC, int G, cudaStream_t stream,
                                const float* dW1_last = nullptr, const float* db1_last = nullptr,
                                const float* dW2_last = nullptr, const float* db2_last = nullptr);
}  // namespace tb

namespace tb {
cudaError_t launch_gate_forward(const void* res, const void* s, const float* a_text, const float* a_video, void* out,
                                void* rev, int B, int L, int E, int text_len, int num_chunks, int perm_s,
                                cudaStream_t stream);
cudaError_t launch_gate_backward(const void* dout, const void* drev, const void* s, const float* a_text,
                                 const float* a_video, void* dres, void* ds, float* da_text, float* da_video, int B,
                                 int L, int E, int text_len, int num_chunks, int perm_s, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_linear_forward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                  const float* ln_b, const float* W1, const float* b1, float* W1c, float* b1c,
                                  float* W1o, float* b1o, void* Out, int B, int H, int NC, int ckpt_group,
                                  cudaStream_t stream);
struct LinearImages;  // recompute_ring.cuh
cudaError_t launch_linear_trajectory(const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                     const float* ln_b, const float* W1s, const float* b1s, long long w_stride,
                                     long long b_stride, const LinearImages& out, int img_slots, int B, int H, int NC,
                                     int t0, int nsteps, cudaStream_t stream);
size_t linear_backward_workspace_bytes(int B, int H, int NC, int G);
cudaError_t launch_linear_backward(const void* XQ, const void* XK, const void* XV, const void* last_eta, const float* ln_w,
                                   const float* ln_b, const float* W1c, const float* b1c, const void* dOut, float* dlnw,
                                   float* dlnb, float* dW1, float* db1, float* dEta, void* dXQ, void* dXK, void* dXV,
                                   void* workspace, size_t workspace_bytes, int B, int H, int NC, int G,
                                   cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_attention_forward(const void* Q, const void* K, const void* V, void* Out, float* lse2, int B, int T,
                                     int H, float scale, cudaStream_t stream);
cudaError_t launch_attention_backward(const void* Q, const void* K, const void* V, const void* Out, const void* dOut,
                                      const float* lse2, float* delta, void* dQ, void* dK, void* dV, int B, int T, int H,
                                      float scale, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_mlp_backward_q(const CUtensorMap& tq, const CUtensorMap& tdo, const float* ln_w, const float* ln_b,
                                  const MlpSlot& slot, void* dXQ, int BH, int H, int NC, int G, int t0, int nsteps,
                                  cudaStream_t stream, unsigned* ready = nullptr);
}  // namespace tb

namespace tb {
cudaError_t launch_debug_spin(int blocks, int threads, long long cycles, int mode, int smem_bytes, float* sink,
                              long long sink_floats, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_process_input(const void* xq, const void* xk, const void* xv, const float* lr_logit, const float* cosT,
                                 const float* sinT, const float* ln_w, const float* ln_b, const int* index, void* XQ,
                                 void* XK, void* XV, void* last_eta, int B, int L, int H, int seq_text_length, int mini_batch,
                                 float base_lr, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_process_input_backward(const void* xq, const void* xk, const void* xv, const float* lr_logit,
                                          const float* cosT, const float* sinT, const float* ln_w, const int* index,
                                          const void* gQ, const void* gK, const void* gV, const float* g_eta, void* gxq,
                                          void* gxk, void* gxv, float* g_logit, float* g_ln_w, float* g_ln_b, int B, int L,
                                          int H, int seq_text_length, int mini_batch, float base_lr, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_output_norm(const void* O, const float* gamma, const float* beta, const int* index, void* out, int B, int L,
                               int H, float eps, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_output_norm_backward(const void* O, const float* gamma, const int* index, const void* gout, void* gO,
                                        float* dgamma, float* dbeta, int B, int L, int H, float eps, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_ln_affine(const void* x, const float* A, const float* C, void* out, int B, int L, int E, int text_len,
                             float eps, cudaStream_t stream);
cudaError_t launch_ln_affine_backward(const void* x, const float* A, const void* gout, void* gx, float* dA, float* dC, int B,
                                      int L, int E, int text_len, float eps, cudaStream_t stream);
cudaError_t launch_gate_add(const void* x, const void* y, const float* G, void* out, int B, int L, int E, int text_len,
                            cudaStream_t stream);
cudaError_t launch_gate_add_backward(const void* gout, const void* y, const float* G, void* dy, float* dG, int B, int L, int E,
                                     int text_len, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_dsmem_probe(int mode, int bytes, int iters, float* out, cudaStream_t stream);
}  // namespace tb

namespace tb {
cudaError_t launch_qk_norm_rope(const void* q, const void* k, const float* gamma, const float* beta, const float* cosT,
                                const float* sinT, void* q_out, void* k_out, int B, int T, int H, int text_len, float eps,
                                cudaStream_t stream);
cudaError_t launch_qk_norm_rope_backward(const void* q, const void* k, const float* gamma, const float* cosT, const float* sinT,
                                         const void* dq_out, const void* dk_out, void* dq, void* dk, float* dgamma, float* dbeta,
                                         int B, int T, int H, int text_len, float eps, cudaStream_t stream);
}  // namespace tb
