// Backward primitives of the training step.  See bwd_kernels.h (status: compiled, not yet run on a B200).
// Specification: oracle/navdp_backward.py (lin_bwd, ln_bwd, gelu_bwd, attn_core_bwd, ...) and oracle/qwen_backward.py.
#include "bwd_kernels.h"

#include <math.h>

#include "dropout.cuh"
#include "n1_ptx.cuh"

namespace n1 {
namespace {

inline int nblk(long n, int t = 256) { return (int)((n + t - 1) / t); }

__device__ __forceinline__ float ldf(const bf16* p) { return __bfloat162float(*p); }

// ---------------------------------------------------------------------------------------------- transpose
__global__ void transpose_kernel(const bf16* __restrict__ in, int rows, int cols, int ld_in, bf16* __restrict__ out,
                                 int ld_out, int rows_pad) {
  __shared__ bf16 tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[(long)r * ld_in + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows_pad) out[(long)c * ld_out + r] = tile[threadIdx.x][i];
  }
}

// ---------------------------------------------------------------------------------------------- column sums
// block = 32 columns x 8 row lanes; blockIdx.y strides over row chunks; partials meet in `out` through atomics
__global__ void colsum_kernel(const bf16* __restrict__ a, const bf16* __restrict__ b, int rows, int cols, int ld_a,
                              int ld_b, float* __restrict__ out, int rows_per_block) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int r_lo = blockIdx.y * rows_per_block, r_hi = min(rows, r_lo + rows_per_block);
  float acc = 0.f;
  if (c < cols)
    for (int r = r_lo + threadIdx.y; r < r_hi; r += 8) {
      const float x = ldf(a + (long)r * ld_a + c);
      acc += b ? x * ldf(b + (long)r * ld_b + c) : x;
    }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    atomicAdd(out + c, t);
  }
}

// ---------------------------------------------------------------------------------------------- norm backward
// one warp per row; statistics recomputed; optional per-row (mean, rstd) written for the parameter-gradient pass
__global__ void norm_bwd_dx_kernel(const bf16* __restrict__ dy, int ld_dy, const bf16* __restrict__ x, int ld_x,
                                   const float* __restrict__ w, const bf16* __restrict__ rg, int ld_rg,
                                   bf16* __restrict__ dx, int ld_dx, float* __restrict__ stats, int rows, int D, float eps,
                                   int rms) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const bf16* xr = x + (long)row * ld_x;
  const bf16* dyr = dy + (long)row * ld_dy;
  float s = 0.f, ss = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float v = ldf(xr + c);
    s += v, ss += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o), ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float mean = rms ? 0.f : s / D;
  const float var = rms ? ss / D : fmaxf(ss / D - mean * mean, 0.f);
  const float rstd = rsqrtf(var + eps);
  if (stats && lane == 0) stats[2 * row] = mean, stats[2 * row + 1] = rstd;
  float g1 = 0.f, g2 = 0.f;  // sum g, sum g * xhat
  for (int c = lane; c < D; c += 32) {
    const float g = ldf(dyr + c) * w[c];
    const float xh = (ldf(xr + c) - mean) * rstd;
    g1 += g, g2 += g * xh;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) g1 += __shfl_xor_sync(0xffffffffu, g1, o), g2 += __shfl_xor_sync(0xffffffffu, g2, o);
  const float m1 = rms ? 0.f : g1 / D, m2 = g2 / D;
  for (int c = lane; c < D; c += 32) {
    const float g = ldf(dyr + c) * w[c];
    const float xh = (ldf(xr + c) - mean) * rstd;
    float r = rstd * (g - m1 - xh * m2);
    if (rg) r += ldf(rg + (long)row * ld_rg + c);
    dx[(long)row * ld_dx + c] = __float2bfloat16(r);
  }
}

__global__ void norm_bwd_param_kernel(const bf16* __restrict__ dy, int ld_dy, const bf16* __restrict__ x, int ld_x,
                                      const float* __restrict__ stats, int rows, int D, float* __restrict__ dw,
                                      float* __restrict__ db, int rows_per_block) {
  __shared__ float rw[8][33], rb[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int r_lo = blockIdx.y * rows_per_block, r_hi = min(rows, r_lo + rows_per_block);
  float aw = 0.f, ab = 0.f;
  if (c < D)
    for (int r = r_lo + threadIdx.y; r < r_hi; r += 8) {
      const float g = ldf(dy + (long)r * ld_dy + c);
      aw += g * (ldf(x + (long)r * ld_x + c) - stats[2 * r]) * stats[2 * r + 1];
      ab += g;
    }
  rw[threadIdx.y][threadIdx.x] = aw, rb[threadIdx.y][threadIdx.x] = ab;
  __syncthreads();
  if (threadIdx.y == 0 && c < D) {
    float tw = 0.f, tb = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tw += rw[i][threadIdx.x], tb += rb[i][threadIdx.x];
    atomicAdd(dw + c, tw);
    if (db) atomicAdd(db + c, tb);
  }
}

// ---------------------------------------------------------------------------------------------- elementwise
__global__ void act_bwd_kernel(const bf16* __restrict__ pre, const bf16* __restrict__ dy, bf16* __restrict__ out, long n,
                               int kind) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = ldf(pre + i), g = ldf(dy + i);
  float d;
  if (kind == ACT_GELU) d = 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x);
  else d = x > 0.f ? 1.f : 0.f;
  out[i] = __float2bfloat16(g * d);
}

__global__ void act_fwd_kernel(const bf16* __restrict__ pre, bf16* __restrict__ out, long n, int kind) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = ldf(pre + i);
  out[i] = __float2bfloat16(kind == ACT_GELU ? 0.5f * x * (1.f + erff(x * 0.70710678118654752f)) : fmaxf(x, 0.f));
}

// ---------------------------------------------------------------------------------------------- dropout (training)
// One Philox block per thread: elements 4g .. 4g + 3 of the site's tensor (dropout.cuh).
// out = (res ? res : 0) + Z y          (dropout_add with a residual; dropout and its backward without)
__global__ void dropout_kernel(const bf16* __restrict__ y, const bf16* __restrict__ res, bf16* __restrict__ out, long n,
                               const DropoutDesc d) {
  const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (4 * g >= n) return;
  const DropKey k = drop_key(d);
  const uint4 w = drop_words(k, (unsigned long long)g);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long e = 4 * g + i;
    if (e >= n) break;
    float v = word_of(w, i) < k.thr ? 0.f : ldf(y + e) * k.scale;
    if (res) v += ldf(res + e);
    out[e] = __float2bfloat16(v);
  }
}

// the keep mask as bytes (tests)
__global__ void dropout_mask_kernel(uint8_t* __restrict__ out, long n, const DropoutDesc d) {
  const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (4 * g >= n) return;
  const DropKey k = drop_key(d);
  const uint4 w = drop_words(k, (unsigned long long)g);
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (4 * g + i < n) out[4 * g + i] = word_of(w, i) < k.thr ? 0 : 1;
}

// activation with dropout after it (the FF inner site): forward out = Z f(pre), backward dpre = Z dy f'(pre)
template <bool BWD>
__global__ void act_dropout_kernel(const bf16* __restrict__ pre, const bf16* __restrict__ dy, bf16* __restrict__ out, long n,
                                   int kind, const DropoutDesc d) {
  const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (4 * g >= n) return;
  const DropKey k = drop_key(d);
  const uint4 w = drop_words(k, (unsigned long long)g);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long e = 4 * g + i;
    if (e >= n) break;
    const float z = word_of(w, i) < k.thr ? 0.f : k.scale;
    const float x = ldf(pre + e);
    float v;
    if (BWD) {
      const float fd = kind == ACT_GELU ? 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x)
                                        : (x > 0.f ? 1.f : 0.f);
      v = z * ldf(dy + e) * fd;
    } else {
      v = z * (kind == ACT_GELU ? 0.5f * x * (1.f + erff(x * 0.70710678118654752f)) : fmaxf(x, 0.f));
    }
    out[e] = __float2bfloat16(v);
  }
}

__global__ void swiglu_bwd_kernel(const bf16* __restrict__ pre, const bf16* __restrict__ dact, bf16* __restrict__ dpre,
                                  long n) {  // n = rows * inter
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float g = ldf(pre + 2 * i), u = ldf(pre + 2 * i + 1), d = ldf(dact + i);
  const float sg = 1.f / (1.f + __expf(-g));
  dpre[2 * i] = __float2bfloat16(d * u * sg * (1.f + g * (1.f - sg)));
  dpre[2 * i + 1] = __float2bfloat16(d * g * sg);
}

__global__ void scale_cols_kernel(const bf16* __restrict__ x, int ld_x, const float* __restrict__ gamma,
                                  const bf16* __restrict__ add, int ld_add, bf16* __restrict__ out, int ld_out, long rows,
                                  int cols) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const long r = i / cols;
  const int c = i % cols;
  float v = ldf(x + r * ld_x + c) * gamma[c];
  if (add) v += ldf(add + r * ld_add + c);
  out[r * ld_out + c] = __float2bfloat16(v);
}

// y = x c + rot_half(x) s  (rot_half(x) = [-x2, x1])  =>  x_bar = y_bar c - rot_half(y_bar s):
//   x1_bar = y1_bar c + y2_bar s ;  x2_bar = y2_bar c - y1_bar s      (c, s shared by the two halves)
__global__ void rope_t_kernel(bf16* __restrict__ x, int ld, const float2* __restrict__ cs, long rows, int heads, int half) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long per_row = (long)heads * half;
  if (i >= rows * per_row) return;
  const long r = i / per_row;
  const int h = (i % per_row) / half, j = i % half;
  bf16* p = x + r * ld + (long)h * 2 * half + j;
  const float2 c = cs[r * half + j];
  const float y1 = ldf(p), y2 = ldf(p + half);
  p[0] = __float2bfloat16(y1 * c.x + y2 * c.y);
  p[half] = __float2bfloat16(y2 * c.x - y1 * c.y);
}

__global__ void adamw_kernel(float* __restrict__ master, bf16* __restrict__ working, const float* __restrict__ grad,
                             float* __restrict__ m, float* __restrict__ v, long n, float lr, float b1, float b2, float eps,
                             float wd, float bc1, float bc2) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float g = grad[i];
  float p = master[i];
  p *= 1.f - lr * wd;                                   // decoupled weight decay first, as torch.optim.AdamW does
  const float mi = b1 * m[i] + (1.f - b1) * g;
  const float vi = b2 * v[i] + (1.f - b2) * g * g;
  m[i] = mi, v[i] = vi;
  p -= (lr / bc1) * mi / (sqrtf(vi) / sqrtf(bc2) + eps);
  master[i] = p;
  if (working) working[i] = __float2bfloat16(p);
}


// ---------------------------------------------------------------------------------------------- small fp32 product
// C[M, N] (+)= op(A) op(B) in fp32 on the CUDA cores, 32 x 32 tiles.  For the products of the training step that are too
// narrow for a tensor-core tile or must stay in fp32: the 3-wide action embedding / action head (navdp.py L79, L186) and
// their gradients, and the position-table resample R [256, 1369] of the DINOv2 ViT and its transpose (dinov2.py L180-211).
__global__ void sgemm_small_kernel(const float* __restrict__ A, int lda, int ta, const float* __restrict__ B, int ldb, int tb,
                                   float* __restrict__ C, int ldc, int M, int N, int K, int accumulate) {
  __shared__ float sa[32][33], sb[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int row = blockIdx.y * 32 + ty, col = blockIdx.x * 32 + tx;
  float acc = 0.f;
  for (int k0 = 0; k0 < K; k0 += 32) {
    {  // sa[ty][tx] = op(A)[row0 + ty, k0 + tx]
      const int r = blockIdx.y * 32 + ty, k = k0 + tx;
      sa[ty][tx] = (r < M && k < K) ? (ta ? A[(long)k * lda + r] : A[(long)r * lda + k]) : 0.f;
    }
    {  // sb[ty][tx] = op(B)[k0 + ty, col0 + tx]
      const int k = k0 + ty, c = blockIdx.x * 32 + tx;
      sb[ty][tx] = (k < K && c < N) ? (tb ? B[(long)c * ldb + k] : B[(long)k * ldb + c]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 32; ++k) acc += sa[ty][k] * sb[k][tx];
    __syncthreads();
  }
  if (row < M && col < N) {
    float* c = C + (long)row * ldc + col;
    *c = accumulate ? *c + acc : acc;
  }
}

// ---------------------------------------------------------------------------------------------- attention backward
constexpr int AQ = 8;  // query rows per tile

// One CTA per (kv sequence, kv head): it alone updates that head's dK / dV rows, looping over the query sequences that
// share the K/V sequence (kv_div), the query heads of the GQA group and the query tiles.  128 threads.
// `stage`: K and V of the head are first copied into shared memory (bf16, rows padded by one word): every pass below reads
// them ~(query heads of the group) x (query tiles) times, and the score / dP passes walk them one key per thread -- from
// global memory those are 2-byte loads 32 rows apart (profiles/r2_launches_ddp_train_v1_summary.txt: 2.5 ms per launch in the
// System-2 backward, 7 query heads x 304 keys x 128).
// DROP: dropout on the probabilities (fixed-length MHA only): dV = (P o Z)^T dO, dS = P o ((dO V^T) o Z - D) with the
// unchanged D = rowsum(dO o O) -- the identity is written out in attention_bwd_mma.cu.
template <bool DROP>
__global__ void __launch_bounds__(128) attn_bwd_kernel(const AttnBwdParams p, const int stage) {
  extern __shared__ float sm[];
  const AttnParams& f = p.f;
  const int hd = f.hd;
  const int kb = blockIdx.x, hk = blockIdx.y;
  const int group = f.heads_q / f.heads_kv;
  const int k_start = f.k_len ? kb * f.k_slot : (f.cu_k ? f.cu_k[kb] : kb * f.seq_k);
  const int sk = f.k_len ? f.k_len[kb] : (f.cu_k ? f.cu_k[kb + 1] - k_start : f.seq_k);
  float* sQ = sm;                    // [AQ][hd]
  float* sDO = sQ + AQ * hd;         // [AQ][hd]
  float* sD = sDO + AQ * hd;         // [AQ]  D_i = do_i . o_i ; then row max, row sum scratch
  float* sM = sD + AQ;
  float* sL = sM + AQ;
  float* sP = sL + AQ;               // [AQ][skp]
  const int skp = (sk + 3) & ~3;
  float* sS = sP + AQ * skp;         // [AQ][skp]  scaled dS
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bf16* gk = f.k + (long)k_start * f.ldk + hk * hd;
  const bf16* gv = f.v + (long)k_start * f.ldv + hk * hd;
  const int hdp = hd + 2;            // padded row (bf16 elements): consecutive keys fall into consecutive banks
  bf16* sK16 = reinterpret_cast<bf16*>(sS + AQ * skp);
  bf16* sV16 = sK16 + (size_t)(stage ? sk : 0) * hdp;
  if (stage) {
    for (int i = tid; i < sk * (hd / 2); i += 128) {
      const int j = i / (hd / 2), c = i % (hd / 2);
      *reinterpret_cast<uint32_t*>(sK16 + j * hdp + 2 * c) = *reinterpret_cast<const uint32_t*>(gk + (long)j * f.ldk + 2 * c);
      *reinterpret_cast<uint32_t*>(sV16 + j * hdp + 2 * c) = *reinterpret_cast<const uint32_t*>(gv + (long)j * f.ldv + 2 * c);
    }
  }
  auto Kat = [&](int j, int d) { return stage ? __bfloat162float(sK16[j * hdp + d]) : ldf(gk + (long)j * f.ldk + d); };
  auto Vat = [&](int j, int d) { return stage ? __bfloat162float(sV16[j * hdp + d]) : ldf(gv + (long)j * f.ldv + d); };
  const int kvd = f.heads_kv * hd;
  float* gdk = p.dk + (long)k_start * kvd + hk * hd;
  float* gdv = p.dv + (long)k_start * kvd + hk * hd;

  for (int b = kb * f.kv_div; b < (kb + 1) * f.kv_div && b < f.batch; ++b) {
    const int q_start = f.cu_q ? f.cu_q[b] : b * f.seq_q;
    const int sq = f.cu_q ? f.cu_q[b + 1] - q_start : f.seq_q;
    const int causal_off = sk - sq;
    for (int hq = 0; hq < group; ++hq) {
      const int h = hk * group + hq;
      for (int q0 = 0; q0 < sq; q0 += AQ) {
        const int nq = min(AQ, sq - q0);
        __syncthreads();
        for (int i = tid; i < AQ * hd; i += 128) {
          const int r = i / hd, d = i % hd;
          const long row = q_start + q0 + r;
          sQ[i] = r < nq ? ldf(f.q + row * f.ldq + h * hd + d) : 0.f;
          sDO[i] = r < nq ? ldf(p.dout + row * p.lddo + h * hd + d) : 0.f;
        }
        __syncthreads();
        if (tid < AQ) {
          float acc = 0.f;
          if (tid < nq)
            for (int d = 0; d < hd; ++d) acc += sDO[tid * hd + d] * ldf(f.o + (long)(q_start + q0 + tid) * f.ldo + h * hd + d);
          sD[tid] = acc;
        }
        // scores
        for (int j = tid; j < sk; j += 128) {
          float acc[AQ];
#pragma unroll
          for (int r = 0; r < AQ; ++r) acc[r] = 0.f;
          for (int d = 0; d < hd; ++d) {
            const float kv = Kat(j, d);
#pragma unroll
            for (int r = 0; r < AQ; ++r) acc[r] += sQ[r * hd + d] * kv;
          }
#pragma unroll
          for (int r = 0; r < AQ; ++r) {
            const bool vis = r < nq && (!f.causal || j <= q0 + r + causal_off);
            sP[r * skp + j] = vis ? acc[r] * f.scale : -INFINITY;
          }
        }
        __syncthreads();
        // row max / sum: warp w owns rows 2w, 2w + 1
        for (int r = warp * 2; r < warp * 2 + 2; ++r) {
          float mx = -INFINITY;
          for (int j = lane; j < sk; j += 32) mx = fmaxf(mx, sP[r * skp + j]);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          float l = 0.f;
          for (int j = lane; j < sk; j += 32) l += mx == -INFINITY ? 0.f : __expf(sP[r * skp + j] - mx);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
          if (lane == 0) sM[r] = mx, sL[r] = l;
        }
        __syncthreads();
        // probabilities, dP = dO V^T, dS = P (dP - D) * scale
        DropKey zk;
        unsigned long long e0 = 0;   // dropout element index of (query q0, key 0)
        if constexpr (DROP) {
          zk = drop_key(f.drop);
          e0 = ((unsigned long long)(b * f.heads_q + h) * sq + q0) * sk;
        }
        for (int j = tid; j < sk; j += 128) {
          float dp[AQ];
#pragma unroll
          for (int r = 0; r < AQ; ++r) dp[r] = 0.f;
          for (int d = 0; d < hd; ++d) {
            const float vv = Vat(j, d);
#pragma unroll
            for (int r = 0; r < AQ; ++r) dp[r] += sDO[r * hd + d] * vv;
          }
#pragma unroll
          for (int r = 0; r < AQ; ++r) {
            const float s = sP[r * skp + j];
            const float pr = (sL[r] > 0.f && s != -INFINITY) ? __expf(s - sM[r]) / sL[r] : 0.f;
            if constexpr (DROP) {
              const float z = r < nq ? drop_mul(zk, e0 + (unsigned long long)r * sk + j) : 0.f;
              sP[r * skp + j] = pr * z;
              sS[r * skp + j] = pr * (dp[r] * z - sD[r]) * f.scale;
            } else {
              sP[r * skp + j] = pr;
              sS[r * skp + j] = pr * (dp[r] - sD[r]) * f.scale;
            }
          }
        }
        __syncthreads();
        // dQ[r, d] = sum_j dS[r, j] K[j, d]
        for (int i = tid; i < nq * hd; i += 128) {
          const int r = i / hd, d = i % hd;
          float acc = 0.f;
          for (int j = 0; j < sk; ++j) acc += sS[r * skp + j] * Kat(j, d);
          p.dq[(long)(q_start + q0 + r) * p.lddq + h * hd + d] = __float2bfloat16(acc);
        }
        // dK[j, d] += sum_r dS[r, j] Q[r, d] ;  dV[j, d] += sum_r P[r, j] dO[r, d]
        for (int i = tid; i < sk * hd; i += 128) {
          const int j = i / hd, d = i % hd;
          float ak = 0.f, av = 0.f;
#pragma unroll
          for (int r = 0; r < AQ; ++r) ak += sS[r * skp + j] * sQ[r * hd + d], av += sP[r * skp + j] * sDO[r * hd + d];
          gdk[(long)j * kvd + d] += ak;
          gdv[(long)j * kvd + d] += av;
        }
      }
    }
  }
}

}  // namespace

void transpose_bf16(const bf16* in, int rows, int cols, int ld_in, bf16* out, int ld_out, int rows_pad, cudaStream_t s) {
  N1_CHECK(rows_pad >= rows && ld_out >= rows_pad, "transpose_bf16: rows_pad / ld_out too small");
  dim3 grid((cols + 31) / 32, (rows_pad + 31) / 32);
  transpose_kernel<<<grid, dim3(32, 8), 0, s>>>(in, rows, cols, ld_in, out, ld_out, rows_pad);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

void colsum_bf16(const bf16* a, const bf16* b, int rows, int cols, int ld_a, int ld_b, float* out, int accumulate,
                 cudaStream_t s) {
  if (!accumulate) N1_CUDA(cudaMemsetAsync(out, 0, (size_t)cols * sizeof(float), s));
  if (rows <= 0) return;
  const int per = 2048;
  dim3 grid((cols + 31) / 32, (rows + per - 1) / per);
  colsum_kernel<<<grid, dim3(32, 8), 0, s>>>(a, b, rows, cols, ld_a, ld_b, out, per);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

// stats scratch: the caller-owned workspace is avoided by a small static pool per call size -- training steps reuse shapes
void norm_bwd(const bf16* dy, int ld_dy, const bf16* x, int ld_x, const float* w, const bf16* rg, int ld_rg, bf16* dx,
              int ld_dx, float* dw, float* db, int rows, int D, float eps, int rms, int accumulate, cudaStream_t s) {
  N1_CHECK(rows > 0 && D > 0 && w != nullptr, "norm_bwd: bad arguments");
  float* stats = nullptr;
  if (dw) N1_CUDA(cudaMallocAsync(&stats, (size_t)rows * 2 * sizeof(float), s));
  norm_bwd_dx_kernel<<<nblk(rows, 8), 256, 0, s>>>(dy, ld_dy, x, ld_x, w, rg, ld_rg, dx, ld_dx, stats, rows, D, eps, rms);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
  if (dw) {
    if (!accumulate) {
      N1_CUDA(cudaMemsetAsync(dw, 0, (size_t)D * sizeof(float), s));
      if (db) N1_CUDA(cudaMemsetAsync(db, 0, (size_t)D * sizeof(float), s));
    }
    const int per = 2048;
    dim3 grid((D + 31) / 32, (rows + per - 1) / per);
    norm_bwd_param_kernel<<<grid, dim3(32, 8), 0, s>>>(dy, ld_dy, x, ld_x, stats, rows, D, dw, db, per);
    prof_count_launch();
    N1_CUDA(cudaGetLastError());
    N1_CUDA(cudaFreeAsync(stats, s));
  }
}

void act_fwd(const bf16* pre, bf16* out, long n, int kind, cudaStream_t s) {
  N1_CHECK(kind == ACT_GELU || kind == ACT_RELU, "act_fwd: GELU or ReLU");
  act_fwd_kernel<<<nblk(n), 256, 0, s>>>(pre, out, n, kind);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void act_bwd(const bf16* pre, const bf16* dy, bf16* out, long n, int kind, cudaStream_t s) {
  N1_CHECK(kind == ACT_GELU || kind == ACT_RELU, "act_bwd: GELU or ReLU");
  act_bwd_kernel<<<nblk(n), 256, 0, s>>>(pre, dy, out, n, kind);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void dropout_apply(const bf16* y, const bf16* res, bf16* out, long n, const DropoutDesc& d, cudaStream_t s) {
  N1_CHECK(d.rng && y && out && n >= 0, "dropout: bad arguments");
  if (n == 0) return;
  dropout_kernel<<<nblk((n + 3) / 4), 256, 0, s>>>(y, res, out, n, d);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void dropout_mask(uint8_t* out, long n, const DropoutDesc& d, cudaStream_t s) {
  N1_CHECK(d.rng && out && n >= 0, "dropout_mask: bad arguments");
  if (n == 0) return;
  dropout_mask_kernel<<<nblk((n + 3) / 4), 256, 0, s>>>(out, n, d);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void act_fwd_dropout(const bf16* pre, bf16* out, long n, int kind, const DropoutDesc& d, cudaStream_t s) {
  N1_CHECK(kind == ACT_GELU || kind == ACT_RELU, "act_fwd: GELU or ReLU");
  N1_CHECK(d.rng, "act_fwd_dropout: no RNG state");
  act_dropout_kernel<false><<<nblk((n + 3) / 4), 256, 0, s>>>(pre, nullptr, out, n, kind, d);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void act_bwd_dropout(const bf16* pre, const bf16* dy, bf16* out, long n, int kind, const DropoutDesc& d, cudaStream_t s) {
  N1_CHECK(kind == ACT_GELU || kind == ACT_RELU, "act_bwd: GELU or ReLU");
  N1_CHECK(d.rng, "act_bwd_dropout: no RNG state");
  act_dropout_kernel<true><<<nblk((n + 3) / 4), 256, 0, s>>>(pre, dy, out, n, kind, d);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void swiglu_bwd(const bf16* pre, const bf16* dact, bf16* dpre, long rows, int inter, cudaStream_t s) {
  swiglu_bwd_kernel<<<nblk(rows * inter), 256, 0, s>>>(pre, dact, dpre, rows * inter);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void scale_cols(const bf16* x, int ld_x, const float* gamma, const bf16* add, int ld_add, bf16* out, int ld_out, long rows,
                int cols, cudaStream_t s) {
  scale_cols_kernel<<<nblk(rows * cols), 256, 0, s>>>(x, ld_x, gamma, add, ld_add, out, ld_out, rows, cols);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void rope_transposed(bf16* x, int ld, const float2* cs, long rows, int heads, int hd, cudaStream_t s) {
  rope_t_kernel<<<nblk(rows * heads * (hd / 2)), 256, 0, s>>>(x, ld, cs, rows, heads, hd / 2);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}
void adamw_step(float* master, bf16* working, const float* grad, float* m, float* v, long n, float lr, float beta1,
                float beta2, float eps, float weight_decay, int step, cudaStream_t s) {
  N1_CHECK(step >= 1, "adamw_step: step counts from 1");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adamw_kernel<<<nblk(n), 256, 0, s>>>(master, working, grad, m, v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}


void sgemm_small(const float* A, int lda, int trans_a, const float* B, int ldb, int trans_b, float* C, int ldc, int M, int N,
                 int K, int accumulate, cudaStream_t s) {
  N1_CHECK(A && B && C && M > 0 && N > 0 && K > 0, "sgemm_small: bad arguments");
  dim3 grid((N + 31) / 32, (M + 31) / 32);
  sgemm_small_kernel<<<grid, dim3(32, 32), 0, s>>>(A, lda, trans_a, B, ldb, trans_b, C, ldc, M, N, K, accumulate);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

void attention_bwd(const AttnBwdParams& p, cudaStream_t s) {
  const AttnParams& f = p.f;
  if (attention_bwd_mma_supported(p)) {
    attention_bwd_mma(p, s);
    return;
  }
  N1_CHECK(f.batch > 0 && f.heads_kv > 0 && f.heads_q % f.heads_kv == 0 && f.kv_div >= 1, "attention_bwd: bad head counts");
  N1_CHECK(f.hd <= 128 && p.dq && p.dk && p.dv && p.dout && f.o, "attention_bwd: null buffers / head_dim > 128");
  N1_CHECK(f.batch % f.kv_div == 0, "attention_bwd: batch must be a multiple of kv_div");
  const int max_sk = f.k_len ? f.k_slot : (f.cu_k ? f.seq_k /* caller passes the maximum here */ : f.seq_k);
  N1_CHECK(max_sk > 0 && max_sk <= 2048, "attention_bwd: key length must be in (0, 2048] (pass the maximum in seq_k)");
  const int skp = (max_sk + 3) & ~3;
  size_t smem = (size_t)(2 * AQ * f.hd + 3 * AQ + 2 * AQ * skp) * sizeof(float);
  // K / V of one head staged in shared memory when they fit next to the tiles (even head_dim, 4-byte aligned rows)
  const size_t kv_bytes = (size_t)2 * max_sk * (f.hd + 2) * sizeof(bf16);
  const bool aligned = f.hd % 2 == 0 && f.ldk % 2 == 0 && f.ldv % 2 == 0 && (reinterpret_cast<uintptr_t>(f.k) & 3) == 0 &&
                       (reinterpret_cast<uintptr_t>(f.v) & 3) == 0;
  const int stage = aligned && smem + kv_bytes <= 200 * 1024 ? 1 : 0;
  if (stage) smem += kv_bytes;
  dim3 grid(f.batch / f.kv_div, f.heads_kv);
  if (f.drop.rng) {
    N1_CHECK(!f.cu_q && !f.cu_k && !f.k_len && f.kv_div == 1 && f.heads_q == f.heads_kv,
             "attention_bwd: dropout needs fixed-length multi-head attention, kv_div 1");
    static size_t attr_d = 0;
    if (smem > attr_d) {
      N1_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_d = smem;
    }
    attn_bwd_kernel<true><<<grid, 128, smem, s>>>(p, stage);
    prof_count_launch();
    N1_CUDA(cudaGetLastError());
    return;
  }
  static size_t attr = 0;
  if (smem > attr) {
    N1_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  attn_bwd_kernel<false><<<grid, 128, smem, s>>>(p, stage);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

}  // namespace n1
