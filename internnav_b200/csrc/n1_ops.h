// Internal C++ interface between the model executors and the kernel launchers (not part of the C ABI).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdexcept>
#include <string>

namespace n1 {

typedef __nv_bfloat16 bf16;

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define N1_CHECK(cond, msg)                                                                       \
  do {                                                                                            \
    if (!(cond)) throw ::n1::Error(-2, std::string(__FILE__) + ":" + std::to_string(__LINE__) + \
                                           ": " + (msg));                                         \
  } while (0)

#define N1_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      throw ::n1::Error(-3, std::string(__FILE__) + ":" + std::to_string(__LINE__) + ": " + #call + \
                                ": " + cudaGetErrorString(e__));                                   \
  } while (0)

// ------------------------------------------------------------------------------------------- GEMM
// out[M, N'] = epilogue(A[M,K] @ W[N,K]^T).  A and W are bf16, K-major (row-major with leading
// dimensions lda / ldw in elements, multiples of 8).  Accumulation in fp32 (TMEM).
enum GemmAct { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2, ACT_SWIGLU = 3, ACT_GELU_TANH = 4, ACT_SILU = 5 };

struct GemmEpilogue {
  const float* bias = nullptr;      // [N]
  const float* gamma = nullptr;     // [N]   layer-scale applied to (acc + bias) after activation
  const bf16* residual = nullptr;   // [M, ldr] added last
  int ldr = 0;
  int act = ACT_NONE;               // ACT_SWIGLU: W rows interleaved (gate_j, up_j); N' = N / 2
  int out_fp32 = 0;                 // write fp32 instead of bf16
  // optional row remap of the OUTPUT (used to drop a patch-GEMM straight into a [n, 1+P, D] token buffer):
  // out_row = (row / rows_per_group) * group_stride + row % rows_per_group + group_offset
  int rows_per_group = 0, group_stride = 0, group_offset = 0;
  const float* row_add = nullptr;   // [rows_per_group, N] fp32 added per (row % rows_per_group) (pos-embed)
};

void gemm_bf16(const bf16* A, int lda, const bf16* W, int ldw, void* out, int ldo, int M, int N, int K,
               const GemmEpilogue& epi, cudaStream_t stream);

int device_sm_count();

// 2-D bf16 tensor map over a row-major [rows, cols] matrix (leading dimension ld elements); box = [box_rows, box_cols];
// operand tiles use box_cols = 64 with the 128-byte swizzle, output staging tiles are unswizzled.
CUtensorMap tma_map_2d(const bf16* ptr, long rows, long cols, long ld, int box_rows, int box_cols, bool swizzle);
void prof_count_gemm(double flops);  // launch + FLOP accounting for GEMM-class kernels outside gemm_tcgen05.cu

// Launch accounting (always on) and optional per-GEMM event timing (bench.py's roofline pass).
struct ProfStats {
  double gemm_ms = 0, gemm_flops = 0;
  long gemm_launches = 0, total_launches = 0;
};
void prof_enable(bool on);
void prof_count_launch(int n = 1);
int prof_begin(double flops, int M, int N, int K, cudaStream_t s);  // event bracket of a GEMM-class kernel (prof on)
void prof_end(int ticket, cudaStream_t s);
ProfStats prof_read_and_reset();
// per-shape sums of the event-timed GEMM launches accumulated by prof_read_and_reset(); clears the table; returns rows
int prof_read_shapes(int* mnk, long* count, double* ms, int cap);

// ------------------------------------------------------------------------------------------- norms
// y = LayerNorm(x) * w + b  (rms=0)   or   y = x / rms(x) * w  (rms=1);  one warp per row; D % 8 == 0.
void layernorm(const bf16* x, int ldx, bf16* y, int ldy, const float* w, const float* b, int rows, int D,
               float eps, int rms, cudaStream_t stream);

// ------------------------------------------------------------------------------------------- dropout
// One dropout site of the training step (mask contract: dropout.cuh).  rng == nullptr: no dropout.
struct DropoutDesc {
  const uint32_t* rng = nullptr;  // device {seed_lo, seed_hi, step, rank}
  float p = 0.f;
  uint32_t thr = 0;               // floor(p * 2^32)
  float scale = 1.f;              // float(1 / (1 - p))
  int site = 0;                   // site id (internnav_b200/dropout.py), < 2^16
};
inline DropoutDesc make_dropout(const void* rng, int site, double p) {
  if (!(p >= 0.0 && p < 1.0) || site < 0 || site >= 65536) throw Error(-2, "dropout: p must be in [0, 1), site in [0, 2^16)");
  DropoutDesc d;
  if (p == 0.0) return d;
  if (!rng) throw Error(-2, "dropout: p > 0 needs the device RNG state");
  d.rng = static_cast<const uint32_t*>(rng), d.p = (float)p, d.site = site;
  d.thr = (uint32_t)(p * 4294967296.0);
  d.scale = (float)(1.0 / (1.0 - p));
  return d;
}

// ------------------------------------------------------------------------------------------- attention
// The sequence description the forward kernels without dropout take by value (kept apart from the dropout fields so that
// their parameter block, and with it their code, stays as it was).
struct AttnCore {
  const bf16* q;  // element (row, head, d) at q[row * ldq + head * hd + d]
  const bf16* k;
  const bf16* v;
  bf16* o;
  int ldq, ldk, ldv, ldo;
  int heads_q, heads_kv, hd;
  int batch;             // number of query sequences
  int seq_q, seq_k;      // fixed lengths when cu_seqlens_* are null
  const int* cu_q;       // [batch + 1] int32 device, optional (varlen)
  const int* cu_k;       // [batch_kv + 1]
  int kv_div;            // query sequence b reads kv sequence b / kv_div (>= 1)
  int causal;            // bottom-right aligned causal mask (key j visible to query i iff j <= i + seq_k - seq_q)
  float scale;
  int max_seq_q;         // upper bound on query length (grid sizing) when varlen
  const int* k_len;      // optional [batch_kv] device: slotted K/V (a KV cache) -- sequence kb occupies rows
  int k_slot;            //   [kb * k_slot, kb * k_slot + k_len[kb]); overrides cu_k / seq_k
  long total_rows;       // optional: rows of the packed q / k / v buffers (var-len self-attention); > 0 lets head_dim 128
                         //   sequences of <= 320 tokens take the tcgen05 kernel (attention_tc.cu), which needs it for TMA
};
struct AttnParams : AttnCore {
  DropoutDesc drop;      // dropout on the probabilities (training): fixed-length MHA with head_dim 48 only; off by default
};
void attention(const AttnParams& p, cudaStream_t stream);
// tcgen05 / TMEM / TMA attention for head_dim 128, var-len self-attention with <= 320 keys per sequence (attention_tc.cu)
bool attention_tc_supported(const AttnParams& p);
void attention_tc128(const AttnParams& p, cudaStream_t stream);

// ------------------------------------------------------------------------------------------- fused decoder blocks
// FF block of the NavDP decoder layer in one kernel (ff_block.cu): out = x + W2 GELU(W1 LayerNorm(x) + b1) + b2 with the
// residual stream held in tensor memory.  x / out bf16 [M, ld] (may alias), w1 [1536, 384], w2 [384, 1536] contiguous.
void ff_block_384(const bf16* x, int ldx, const float* ln_w, const float* ln_b, float eps, const bf16* w1, const float* b1,
                  const bf16* w2, const float* b2, bf16* out, int ldo, int M, int cluster, cudaStream_t stream);

// ------------------------------------------------------------------------------------------- NextDiT rows (nextdit_kernels.cu)
// Modulated / gated norms of LuminaNextDiTBlock (nextdit_traj.py L125-178) over bf16 rows of width D <= 1024, D % 8 == 0;
// `mod` holds one vector per group of `rows_per_group` consecutive rows (row stride ld_mod), or is null:
//   mode 0: out = RMSNorm(x) * w * (1 + mod[g])     mode 1: out = LayerNorm_noaffine(x) * (1 + mod[g])
//   mode 2: out = res + tanh(mod[g]) * RMSNorm(x) * w
void mod_norm(const bf16* x, int ldx, const float* w, const bf16* mod, int ld_mod, int rows_per_group, const bf16* res, int ldr,
              bf16* out, int ldo, long rows, int D, float eps, int mode, cudaStream_t stream);
void add_bf16(const bf16* a, const bf16* b, bf16* out, long n, cudaStream_t stream);
// action_encoder + positional code (internvla_n1.py L401-409): lat fp32 [rows, 3] -> bf16 [rows, D]; pos fp32 [T, D]
void action_embed(const float* lat, const float* w, const float* b, const float* pos, bf16* out, long rows, int T, int D,
                  cudaStream_t stream);
// classifier-free guidance + flow-matching Euler update (internvla_n1.py L422-427): pred bf16 [2n or n, ld], lat fp32 [n, 3]
void cfg_euler(const bf16* pred, int ld, long n, int cfg, float scale, float dt, float* lat, cudaStream_t stream);

// ------------------------------------------------------------------------------------------- action tail (postprocess.cu)
// traj fp32 [B * Ns, T, 3] (sampler output, un-normalised) -> ids int32 [B, cap] (zero padded), count int32 [B] (ids the
// walk produced; may exceed cap), optional mean path double [B, T + 1, 2].  max_actions > 0: stop once that many ids exist.
void traj_to_actions(const float* traj, int B, int Ns, int T, double turn_rad, double step_size, int lookahead,
                     int max_actions, int cap, int* ids, int* count, double* mean_out, cudaStream_t s);

}  // namespace n1
