// Backward primitives of the training step (SURVEY.md §8 row a13) -- first version, CUDA-core kernels written for
// correctness against oracle/navdp_backward.py and oracle/qwen_backward.py (the hand-written backward specs), not yet
// for speed; the matrix products of the backward (dgrad, wgrad) go through the tcgen05 GEMM on transposed operands.
//
// STATUS: written at the end of round 1 without GPU time left -- compiled for sm_100a, NOT yet run on a B200.  Nothing
// on the inference path calls into this file; the op-level tests (tests/test_bwd_ops_gpu.py) are skipped until a parity
// run is on record.
#pragma once
#include "n1_ops.h"

namespace n1 {

// out[c, r] = in[r, c] for r < rows, zero for rows <= r < rows_pad (rows_pad % 8 == 0 makes `out` a legal GEMM operand
// with K = rows_pad).  in: [rows, ld_in], out: [cols, ld_out >= rows_pad].
void transpose_bf16(const bf16* in, int rows, int cols, int ld_in, bf16* out, int ld_out, int rows_pad, cudaStream_t s);

// out[c] (+)= sum_r a[r, c] * (b ? b[r, c] : 1)   fp32; deterministic (fixed reduction tree).  accumulate: add to out.
void colsum_bf16(const bf16* a, const bf16* b, int rows, int cols, int ld_a, int ld_b, float* out, int accumulate,
                 cudaStream_t s);

// LayerNorm (rms = 0) / RMSNorm (rms = 1) backward, statistics recomputed from x:
//   dx[r, :] = (residual_grad ? residual_grad[r, :] : 0) + rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * w
//   (RMSNorm: xhat = x * rstd, no mean subtraction: dx = rstd * (g - xhat * mean(g * xhat)))
//   dw[c] (+)= sum_r dy * xhat ; db[c] (+)= sum_r dy      (dw / db may be null: frozen norm, e.g. the LLM's)
void norm_bwd(const bf16* dy, int ld_dy, const bf16* x, int ld_x, const float* w, const bf16* residual_grad, int ld_rg,
              bf16* dx, int ld_dx, float* dw, float* db, int rows, int D, float eps, int rms, int accumulate,
              cudaStream_t s);

// Elementwise activation forward (training keeps the pre-activation, so the GEMM epilogue cannot fuse it): out = f(pre)
void act_fwd(const bf16* pre, bf16* out, long n, int kind, cudaStream_t s);
// Elementwise activation backward on the saved pre-activation: out = dy * f'(pre); kind: ACT_GELU (exact erf) / ACT_RELU
void act_bwd(const bf16* pre, const bf16* dy, bf16* out, long n, int kind, cudaStream_t s);
// Dropout of the training step (mask contract: dropout.cuh; d.rng must be set):
//   dropout_apply   out = (res ? res : 0) + Z y   -- a residual branch with dropout, a dropped tensor, or the backward Z dy
//   dropout_mask    out[e] = keep(e) as 0 / 1 bytes (tests)
//   act_*_dropout   the FF inner site: out = Z f(pre) ; dpre = Z dy f'(pre)  (the pre-activation stays the only saved tensor)
void dropout_apply(const bf16* y, const bf16* res, bf16* out, long n, const DropoutDesc& d, cudaStream_t s);
void dropout_mask(uint8_t* out, long n, const DropoutDesc& d, cudaStream_t s);
void act_fwd_dropout(const bf16* pre, bf16* out, long n, int kind, const DropoutDesc& d, cudaStream_t s);
void act_bwd_dropout(const bf16* pre, const bf16* dy, bf16* out, long n, int kind, const DropoutDesc& d, cudaStream_t s);
// SwiGLU backward: pre [R, 2I] interleaved (gate_j, up_j) pre-activations, dact [R, I] -> dpre [R, 2I] interleaved
void swiglu_bwd(const bf16* pre, const bf16* dact, bf16* dpre, long rows, int inter, cudaStream_t s);
// out[r, c] = x[r, c] * gamma[c] (+ add[r, c])   -- layer scale and its backward share this
void scale_cols(const bf16* x, int ld_x, const float* gamma, const bf16* add, int ld_add, bf16* out, int ld_out, long rows,
                int cols, cudaStream_t s);
// Transposed rotate-half rotary: x_bar = y_bar * c - rot_half(y_bar * s), in place on `heads` heads of every row
void rope_transposed(bf16* x, int ld, const float2* cs, long rows, int heads, int hd, cudaStream_t s);

// C[M, N] (+)= op(A) op(B), all fp32 row-major with leading dimensions; trans_a: A is stored [K, M]; trans_b: B is stored
// [N, K].  CUDA-core kernel for the narrow (3-wide) and fp32-only products of the training step.
void sgemm_small(const float* A, int lda, int trans_a, const float* B, int ldb, int trans_b, float* C, int ldc, int M, int N,
                 int K, int accumulate, cudaStream_t s);

// Softmax-attention backward with recomputed probabilities.  Addressing as AttnParams (n1_ops.h): q / k / v / o / do
// element (row, head, d) at ptr[row * ld + head * hd + d]; fixed or var-len / slotted sequences; GQA; bottom-right
// causal.  Outputs: dq bf16 (same addressing as q with lddq), dk / dv fp32 [rows_k, heads_kv * hd] dense, ZEROED by the
// caller when several launches accumulate into them (kv_div > 1: query sequences sharing one K/V sequence).
// f.drop set: the backward of attention with dropout on the probabilities (fixed-length MHA, head_dim 48 on the tensor cores).
struct AttnBwdParams {
  AttnParams f;          // forward description; f.o is the forward output
  const bf16* dout;      // gradient of f.o, same layout (lddo)
  int lddo;
  bf16* dq;
  int lddq;
  float* dk;
  float* dv;             // [rows_k, heads_kv * hd]
};
void attention_bwd(const AttnBwdParams& p, cudaStream_t s);
// Weight gradient dW[No, Ko] (+)= dY[M, No]^T X[M, Ko] without operand transposes (wgrad_tn.cu): both operands read in place
// as MN-major UMMA tiles, the M range split over CTAs, partial tiles summed in a fixed order.  bf16 in, fp32 out.
int wgrad_tn_splits(int M, int No, int Ko);
size_t wgrad_tn_workspace_bytes(int M, int No, int Ko);
void wgrad_tn(const bf16* dy, int ld_dy, const bf16* x, int ld_x, int M, int No, int Ko, float* out, int accumulate, void* ws,
              size_t ws_bytes, cudaStream_t stream);
// tensor-core path (attention_bwd_mma.cu): fixed-length MHA, head_dim 48 / 64, one head's operands within shared memory;
// attention_bwd() takes it whenever it applies (N1_ATTN_BWD_MMA=0 keeps the scalar kernel)
bool attention_bwd_mma_supported(const AttnBwdParams& p);
void attention_bwd_mma(const AttnBwdParams& p, cudaStream_t s);

// Fused AdamW step on fp32 master parameters with a bf16 working copy (torch.optim.AdamW semantics: decoupled decay,
// bias correction): p -= lr * (m_hat / (sqrt(v_hat) + eps) + wd * p)
void adamw_step(float* master, bf16* working, const float* grad, float* m, float* v, long n, float lr, float beta1,
                float beta2, float eps, float weight_decay, int step, cudaStream_t s);

}  // namespace n1
