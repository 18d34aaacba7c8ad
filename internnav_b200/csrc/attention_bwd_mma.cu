// Attention backward on the tensor cores for the trainable System-1 branches (head_dim 48 / 64, fixed-length sequences of
// up to a few hundred tokens): the DINOv2 depth ViT (257 tokens, 6 heads x 64) and the NavDP decoder / RGB-D former
// (8 heads x 48).  Reference: torch autograd through nn.MultiheadAttention / dinov2 Attention in
// internnav/model/basemodel/internvla_n1/navdp.py L291-312 (the loss that is back-propagated), dinov2.py L180-322.
//
// One CTA per (sequence, head), 8 warps.  Q, K, V and dO of that head live in shared memory (bf16, padded rows); the row
// log-sum-exp is recomputed here (the forward kernel does not keep it), so the kernel takes exactly the forward operands.
//   phase 1  D_i = dO_i . O_i                                                (one thread per query row)
//   phase 2  per 16-query block (one warp): LSE over all keys, then dQ = (P o (dP - D)) K * scale     -> global bf16
//   phase 3  per 16-key block (one warp):  dV = P^T dO,  dK = (P o (dP - D))^T Q * scale              -> global fp32
// S = Q K^T is therefore formed three times (7 matmuls instead of the minimal 5) -- in exchange no atomics, no cross-warp
// reductions and a deterministic result.  All products run on mma.sync.m16n8k16 (bf16 operands, fp32 accumulate) with
// ldmatrix operand fetch: the tiles are 16 x 32 per warp, far below what a tcgen05 128-row MMA needs, and the whole
// backward of the depth ViT is ~1.6 TFLOP per step.
//
// DROP (training, dropout on the probabilities; mask Z = keep / (1 - p) of dropout.cuh, recomputed from the element index):
// the forward computed O = (P o Z) V with P = softmax(S).  Then
//   dV = (P o Z)^T dO,   dP = (dO V^T) o Z,   dS = P o (dP - D)  with the unchanged D_i = dO_i . O_i,
// because the softmax backward needs sum_j P_ij dP_ij = sum_j P_ij Z_ij (dO_i . V_j) = dO_i . sum_j (P o Z)_ij V_j = dO_i . O_i.
// Phases 2 and 3 apply Z to the same (query, key) element wherever they re-form S.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>

#include "bwd_kernels.h"
#include "dropout.cuh"
#include "n1_ops.h"

namespace n1 {
namespace {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldsm4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

constexpr int kChunk = 32;   // keys (phase 2) / queries (phase 3) per inner step
constexpr int kWarps = 8;

// rows [0, n_valid) of one head copied into padded shared rows; rows up to n_pad are zeroed
template <int HD>
__device__ __forceinline__ void stage_rows(uint8_t* dst, const bf16* g, long ld, int n_valid, int n_pad) {
  constexpr int RB = HD * 2 + 16, CPR = HD / 8;
  for (int i = threadIdx.x; i < n_pad * CPR; i += blockDim.x) {
    const int r = i / CPR, c = i % CPR;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < n_valid) v = *reinterpret_cast<const uint4*>(g + (long)r * ld + c * 8);
    *reinterpret_cast<uint4*>(dst + r * RB + c * 16) = v;
  }
}

// A-operand fragments (16 rows x HD) of the row block starting at `row0`
template <int HD>
__device__ __forceinline__ void load_a_frags(const uint8_t* s, int row0, int lane, uint32_t (&f)[HD / 16][4]) {
  constexpr int RB = HD * 2 + 16;
  const int lm = lane >> 3, lr = lane & 7;
#pragma unroll
  for (int ks = 0; ks < HD / 16; ++ks)
    ldsm4(smem_addr(s + (row0 + lr + (lm & 1) * 8) * RB + (ks * 16 + (lm >> 1) * 8) * 2), f[ks][0], f[ks][1], f[ks][2], f[ks][3]);
}

// acc[4 n-tiles][4] = A(16 x HD) . B^T, B = 32 rows of `s` starting at row0 (row-major [n][k])
template <int HD>
__device__ __forceinline__ void mm_nt32(float (&acc)[4][4], const uint32_t (&a)[HD / 16][4], const uint8_t* s, int row0, int lane) {
  constexpr int RB = HD * 2 + 16;
  const int lm = lane >> 3, lr = lane & 7;
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < HD / 16; ++ks) {
#pragma unroll
    for (int np = 0; np < 2; ++np) {
      uint32_t b0, b1, b2, b3;
      ldsm4(smem_addr(s + (row0 + np * 16 + (lm >> 1) * 8 + lr) * RB + (ks * 16 + (lm & 1) * 8) * 2), b0, b1, b2, b3);
      mma16816(acc[2 * np], a[ks], b0, b1);
      mma16816(acc[2 * np + 1], a[ks], b2, b3);
    }
  }
}

// acc[HD/8 n-tiles][4] += A(16 x 32, two k-steps of fragments) . B, B = 32 rows of `s` starting at row0 (row-major [k][n])
template <int HD>
__device__ __forceinline__ void mm_nn32(float (&acc)[HD / 8][4], const uint32_t (&a)[2][4], const uint8_t* s, int row0, int lane) {
  constexpr int RB = HD * 2 + 16;
  const int lm = lane >> 3, lr = lane & 7;
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
    for (int np = 0; np < HD / 16; ++np) {
      uint32_t b0, b1, b2, b3;
      ldsm4_t(smem_addr(s + (row0 + kk * 16 + (lm & 1) * 8 + lr) * RB + (np * 16 + (lm >> 1) * 8) * 2), b0, b1, b2, b3);
      mma16816(acc[2 * np], a[kk], b0, b1);
      mma16816(acc[2 * np + 1], a[kk], b2, b3);
    }
  }
}

template <int HD, bool DROP>
__global__ void __launch_bounds__(kWarps * 32, 1) attn_bwd_mma_kernel(AttnBwdParams p, int sqp, int skp) {
  constexpr int RB = HD * 2 + 16, KS = HD / 16, NO = HD / 8;
  const AttnParams& f = p.f;
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sDO = sQ + (size_t)sqp * RB;
  uint8_t* sK = sDO + (size_t)sqp * RB;
  uint8_t* sV = sK + (size_t)skp * RB;
  float* sL = reinterpret_cast<float*>(sV + (size_t)skp * RB);  // [sqp] row log-sum-exp, base 2, of the scaled scores
  float* sD = sL + sqp;                                          // [sqp] dO_i . O_i

  const int b = blockIdx.x, h = blockIdx.y;
  const int sq = f.seq_q, sk = f.seq_k;
  const long q_start = (long)b * sq, k_start = (long)b * sk;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int causal_off = sk - sq;
  const float sl2 = f.scale * 1.4426950408889634f;
  DropKey zk;
  unsigned long long e0 = 0;   // dropout element index of (query 0, key 0) of this (sequence, head)
  if constexpr (DROP) {
    zk = drop_key(f.drop);
    e0 = (unsigned long long)(b * f.heads_q + h) * sq * sk;
  }

  stage_rows<HD>(sQ, f.q + q_start * f.ldq + h * HD, f.ldq, sq, sqp);
  stage_rows<HD>(sDO, p.dout + q_start * p.lddo + h * HD, p.lddo, sq, sqp);
  stage_rows<HD>(sK, f.k + k_start * f.ldk + h * HD, f.ldk, sk, skp);
  stage_rows<HD>(sV, f.v + k_start * f.ldv + h * HD, f.ldv, sk, skp);
  // phase 1: D_i (dO read back from global: the staged copy may not be visible yet)
  for (int i = tid; i < sqp; i += blockDim.x) {
    float acc = 0.f;
    if (i < sq) {
      const bf16* go = f.o + (q_start + i) * f.ldo + h * HD;
      const bf16* gd = p.dout + (q_start + i) * p.lddo + h * HD;
#pragma unroll
      for (int c = 0; c < HD / 8; ++c) {
        const uint4 a = *reinterpret_cast<const uint4*>(go + c * 8), d = *reinterpret_cast<const uint4*>(gd + c * 8);
        const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* pd = reinterpret_cast<const __nv_bfloat162*>(&d);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 x = __bfloat1622float2(pa[e]), y = __bfloat1622float2(pd[e]);
          acc += x.x * y.x + x.y * y.y;
        }
      }
    }
    sD[i] = acc;
  }
  __syncthreads();

  // ---------------------------------------------------------------- phase 2: LSE and dQ, one 16-query block per warp
  for (int rb = warp; rb * 16 < sq; rb += kWarps) {
    uint32_t qf[KS][4], dof[KS][4];
    load_a_frags<HD>(sQ, rb * 16, lane, qf);
    load_a_frags<HD>(sDO, rb * 16, lane, dof);
    const int qa = rb * 16 + (lane >> 2), qb = qa + 8;  // query index of accumulator elements 0/1 and 2/3
    float mrow[2] = {-INFINITY, -INFINITY}, lrow[2] = {0.f, 0.f};
    for (int kc = 0; kc * kChunk < sk; ++kc) {
      float s[4][4];
      mm_nt32<HD>(s, qf, sK, kc * kChunk, lane);
      float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = kc * kChunk + i * 8 + (lane & 3) * 2 + (e & 1);
          const int qi = e < 2 ? qa : qb;
          const bool vis = key < sk && (!f.causal || key <= qi + causal_off);
          s[i][e] = vis ? s[i][e] * sl2 : -INFINITY;
          mx[e >> 1] = fmaxf(mx[e >> 1], s[i][e]);
        }
      }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        const float mnew = fmaxf(mrow[r], mx[r]);
        const float muse = mnew == -INFINITY ? 0.f : mnew;
        float part = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) part += exp2f(s[i][2 * r] - muse) + exp2f(s[i][2 * r + 1] - muse);
        lrow[r] = lrow[r] * exp2f(mrow[r] - muse) + part;   // lrow holds this thread's share; summed over the quad below
        mrow[r] = mnew;
      }
    }
    float lse[2], dd[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      lrow[r] += __shfl_xor_sync(0xffffffffu, lrow[r], 1);
      lrow[r] += __shfl_xor_sync(0xffffffffu, lrow[r], 2);
      lse[r] = lrow[r] > 0.f ? mrow[r] + log2f(lrow[r]) : INFINITY;  // fully masked row: every probability is 0
    }
    if ((lane & 3) == 0) sL[qa] = lse[0], sL[qb] = lse[1];
    dd[0] = sD[qa], dd[1] = sD[qb];

    float dq[NO][4];
#pragma unroll
    for (int i = 0; i < NO; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
    for (int kc = 0; kc * kChunk < sk; ++kc) {
      float s[4][4], dp[4][4];
      mm_nt32<HD>(s, qf, sK, kc * kChunk, lane);
      mm_nt32<HD>(dp, dof, sV, kc * kChunk, lane);
      uint32_t dsf[2][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float ds[4];
        if constexpr (DROP) {
          const int key0 = kc * kChunk + i * 8 + (lane & 3) * 2;
          const float2 za = drop_mul2(zk, e0 + (unsigned long long)qa * sk + key0);
          const float2 zb = drop_mul2(zk, e0 + (unsigned long long)qb * sk + key0);
          dp[i][0] *= za.x, dp[i][1] *= za.y, dp[i][2] *= zb.x, dp[i][3] *= zb.y;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = kc * kChunk + i * 8 + (lane & 3) * 2 + (e & 1);
          const int qi = e < 2 ? qa : qb;
          const bool vis = key < sk && (!f.causal || key <= qi + causal_off);
          const float pr = vis ? exp2f(s[i][e] * sl2 - lse[e >> 1]) : 0.f;
          ds[e] = pr * (dp[i][e] - dd[e >> 1]) * f.scale;
        }
        dsf[i >> 1][(i & 1) * 2 + 0] = pack2(ds[0], ds[1]);
        dsf[i >> 1][(i & 1) * 2 + 1] = pack2(ds[2], ds[3]);
      }
      mm_nn32<HD>(dq, dsf, sK, kc * kChunk, lane);
    }
    bf16* g = p.dq + q_start * p.lddq + h * HD + (lane & 3) * 2;
#pragma unroll
    for (int i = 0; i < NO; ++i) {
      if (qa < sq) *reinterpret_cast<uint32_t*>(g + (long)qa * p.lddq + i * 8) = pack2(dq[i][0], dq[i][1]);
      if (qb < sq) *reinterpret_cast<uint32_t*>(g + (long)qb * p.lddq + i * 8) = pack2(dq[i][2], dq[i][3]);
    }
  }
  __syncthreads();  // sL complete (entries of padding rows >= sq are never used: phase 3 masks them by index)

  // ---------------------------------------------------------------- phase 3: dK and dV, one 16-key block per warp
  const int kvd = f.heads_kv * HD;
  for (int kb = warp; kb * 16 < sk; kb += kWarps) {
    uint32_t kf[KS][4], vf[KS][4];
    load_a_frags<HD>(sK, kb * 16, lane, kf);
    load_a_frags<HD>(sV, kb * 16, lane, vf);
    const int ka = kb * 16 + (lane >> 2), kbb = ka + 8;
    float dk[NO][4], dv[NO][4];
#pragma unroll
    for (int i = 0; i < NO; ++i) dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
    for (int qc = 0; qc * kChunk < sq; ++qc) {
      float st[4][4], dpt[4][4];
      mm_nt32<HD>(st, kf, sQ, qc * kChunk, lane);     // S^T: rows = keys, columns = queries
      mm_nt32<HD>(dpt, vf, sDO, qc * kChunk, lane);   // dP^T
      uint32_t pf[2][4], dsf[2][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int q0 = qc * kChunk + i * 8 + (lane & 3) * 2;
        const float2 l2 = *reinterpret_cast<const float2*>(sL + q0), d2 = *reinterpret_cast<const float2*>(sD + q0);
        float pr[4], ds[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int qi = q0 + (e & 1), key = e < 2 ? ka : kbb;
          const bool vis = key < sk && qi < sq && (!f.causal || key <= qi + causal_off);
          const float l = (e & 1) ? l2.y : l2.x, d = (e & 1) ? d2.y : d2.x;
          pr[e] = vis ? exp2f(st[i][e] * sl2 - l) : 0.f;
          if constexpr (DROP) {   // rows are keys here: the two columns of a pair are Sk elements apart
            const float z = vis ? drop_mul(zk, e0 + (unsigned long long)qi * sk + key) : 0.f;
            ds[e] = pr[e] * (dpt[i][e] * z - d) * f.scale;
            pr[e] *= z;
          } else {
            ds[e] = pr[e] * (dpt[i][e] - d) * f.scale;
          }
        }
        pf[i >> 1][(i & 1) * 2 + 0] = pack2(pr[0], pr[1]);
        pf[i >> 1][(i & 1) * 2 + 1] = pack2(pr[2], pr[3]);
        dsf[i >> 1][(i & 1) * 2 + 0] = pack2(ds[0], ds[1]);
        dsf[i >> 1][(i & 1) * 2 + 1] = pack2(ds[2], ds[3]);
      }
      mm_nn32<HD>(dv, pf, sDO, qc * kChunk, lane);
      mm_nn32<HD>(dk, dsf, sQ, qc * kChunk, lane);
    }
    float* gk = p.dk + k_start * kvd + h * HD + (lane & 3) * 2;
    float* gv = p.dv + k_start * kvd + h * HD + (lane & 3) * 2;
#pragma unroll
    for (int i = 0; i < NO; ++i) {
      if (ka < sk) {
        *reinterpret_cast<float2*>(gk + (long)ka * kvd + i * 8) = make_float2(dk[i][0], dk[i][1]);
        *reinterpret_cast<float2*>(gv + (long)ka * kvd + i * 8) = make_float2(dv[i][0], dv[i][1]);
      }
      if (kbb < sk) {
        *reinterpret_cast<float2*>(gk + (long)kbb * kvd + i * 8) = make_float2(dk[i][2], dk[i][3]);
        *reinterpret_cast<float2*>(gv + (long)kbb * kvd + i * 8) = make_float2(dv[i][2], dv[i][3]);
      }
    }
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <int HD, bool DROP = false>
void launch(const AttnBwdParams& p, int sqp, int skp, size_t smem, cudaStream_t s) {
  static size_t attr = 0;
  if (smem > attr) {
    N1_CUDA(cudaFuncSetAttribute(attn_bwd_mma_kernel<HD, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  attn_bwd_mma_kernel<HD, DROP><<<dim3(p.f.batch, p.f.heads_q), kWarps * 32, smem, s>>>(p, sqp, skp);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

}  // namespace

size_t attention_bwd_mma_smem(const AttnBwdParams& p) {
  const int sqp = (p.f.seq_q + kChunk - 1) / kChunk * kChunk, skp = (p.f.seq_k + kChunk - 1) / kChunk * kChunk;
  return (size_t)(2 * sqp + 2 * skp) * (p.f.hd * 2 + 16) + (size_t)2 * sqp * sizeof(float);
}

// Fixed-length multi-head attention (no GQA, no shared K/V, no slotted cache) with head_dim 48 / 64, 16-byte aligned rows and
// all four operand tiles of one head within the shared memory of an SM.  N1_ATTN_BWD_MMA=0 keeps the scalar kernel.
bool attention_bwd_mma_supported(const AttnBwdParams& p) {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("N1_ATTN_BWD_MMA");
    on = e ? atoi(e) : 1;
  }
  const AttnParams& f = p.f;
  if (!on || (f.hd != 48 && f.hd != 64) || f.heads_q != f.heads_kv || f.kv_div != 1) return false;
  if (f.cu_q || f.cu_k || f.k_len || f.seq_q <= 0 || f.seq_k <= 0) return false;
  if ((f.ldq | f.ldk | f.ldv | f.ldo | p.lddo) % 8 != 0 || p.lddq % 2 != 0) return false;
  if (!aligned16(f.q) || !aligned16(f.k) || !aligned16(f.v) || !aligned16(f.o) || !aligned16(p.dout)) return false;
  if ((reinterpret_cast<uintptr_t>(p.dq) & 3) || (reinterpret_cast<uintptr_t>(p.dk) & 7) || (reinterpret_cast<uintptr_t>(p.dv) & 7))
    return false;
  return attention_bwd_mma_smem(p) <= 220 * 1024;
}

void attention_bwd_mma(const AttnBwdParams& p, cudaStream_t s) {
  N1_CHECK(attention_bwd_mma_supported(p), "attention_bwd_mma: unsupported problem");
  const int sqp = (p.f.seq_q + kChunk - 1) / kChunk * kChunk, skp = (p.f.seq_k + kChunk - 1) / kChunk * kChunk;
  const size_t smem = attention_bwd_mma_smem(p);
  if (p.f.drop.rng) {
    N1_CHECK(p.f.hd == 48, "attention_bwd_mma: dropout needs head_dim 48");
    launch<48, true>(p, sqp, skp, smem, s);
  } else if (p.f.hd == 48)
    launch<48>(p, sqp, skp, smem, s);
  else
    launch<64>(p, sqp, skp, smem, s);
}

}  // namespace n1
