// Scaled-dot-product attention, forward only, bf16 in / bf16 out, fp32 softmax statistics.
//
// One kernel template covers every attention call site on the InternVLA-N1 hot path:
//   * NavDP decoder causal self-attention (T<=32, 8 x hd 48) and cross-attention to the 34 condition tokens shared
//     by the 32 samples of an environment (kv_div = 32)                          -- navdp.py L57-66, L192
//   * goal compressor (1 query x 4 keys)                                          -- navdp_backbone.py L98
//   * DINOv2 ViT-S MHSA (257 tokens, 6 x hd 64)                                   -- dinov2_layers/attention.py L49-62
//   * Q-former self (32) / cross (32 x 1024) attention, 8 x hd 48                 -- navdp_backbone.py L148, L200
//   * Qwen2.5-VL ViT windowed / full varlen attention (16 x hd 80)                -- transformers modeling_qwen2_5_vl.py
//   * Qwen2.5-VL decoder causal GQA prefill (28 q / 4 kv heads, hd 128)           -- idem
//
// Flash-attention style: a CTA owns 64 query rows of one (sequence, head); 4 warps x 16 rows; K/V streamed in
// 64-key tiles through a 2-stage cp.async ring; S = QK^T and O += PV on mma.sync.m16n8k16 (bf16, fp32 accumulate)
// with ldmatrix operand fetch; online softmax in registers with quad shuffles.
// The hd-128 var-len prefill of up to 320 tokens per sequence is routed to the tcgen05 kernel (attention_tc.cu) by
// attention(); this file keeps the general path (any length, GQA, slotted K/V cache, head_dim 48 / 64 / 80 / 128).
#include <stdlib.h>

#include <type_traits>

#include "dropout.cuh"
#include "n1_ops.h"
#include "n1_ptx.cuh"

namespace n1 {
namespace {

constexpr int BQ = 64;
constexpr int BKV = 64;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(sz)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int HD>
struct ACfg {
  static constexpr int kRowBytes = HD * 2 + 16;  // +16 keeps the 8 row addresses of an ldmatrix in distinct banks
  static constexpr int kTileBytes = 64 * kRowBytes;
  static constexpr int kSmemBytes = 5 * kTileBytes;  // Q, K[2], V[2]
};

template <int HD>
__device__ __forceinline__ void load_tile(uint8_t* sdst, const bf16* gbase, long ld, int row0, int nrows_valid) {
  // 64 rows x HD bf16; rows >= nrows_valid are zero-filled.
  constexpr int kChunks = HD / 8;
  for (int c = threadIdx.x; c < 64 * kChunks; c += 128) {
    const int r = c / kChunks, ch = c % kChunks;
    const bool ok = (row0 + r) < nrows_valid;
    const bf16* src = gbase + (long)(ok ? row0 + r : 0) * ld + ch * 8;
    cp_async16(sdst + r * ACfg<HD>::kRowBytes + ch * 16, src, ok);
  }
}

// DROP (training): dropout on the probabilities.  The row sum l is taken over the undropped probabilities and only the P
// operand of O += P V is masked and scaled, so O = (softmax(S) o Z) V with Z the scaled keep mask of dropout.cuh.
template <bool DROP>
using AttnKParams = std::conditional_t<DROP, AttnParams, AttnCore>;

template <int HD, bool DROP>
__global__ void __launch_bounds__(128) attn_kernel(const AttnKParams<DROP> p) {
  using C = ACfg<HD>;
  extern __shared__ __align__(16) uint8_t asmem[];
  uint8_t* sQ = asmem;
  uint8_t* sK = asmem + C::kTileBytes;
  uint8_t* sV = asmem + 3 * C::kTileBytes;

  const int b = blockIdx.z, h = blockIdx.y, qt = blockIdx.x;
  const int q_start = p.cu_q ? p.cu_q[b] : b * p.seq_q;
  const int sq = p.cu_q ? p.cu_q[b + 1] - q_start : p.seq_q;
  const int q0 = qt * BQ;
  if (q0 >= sq) return;
  const int kb = b / p.kv_div;
  const int k_start = p.k_len ? kb * p.k_slot : (p.cu_k ? p.cu_k[kb] : kb * p.seq_k);
  const int sk = p.k_len ? p.k_len[kb] : (p.cu_k ? p.cu_k[kb + 1] - k_start : p.seq_k);
  const int hk = h / (p.heads_q / p.heads_kv);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const bf16* gq = p.q + (long)q_start * p.ldq + h * HD;
  const bf16* gk = p.k + (long)k_start * p.ldk + hk * HD;
  const bf16* gv = p.v + (long)k_start * p.ldv + hk * HD;

  const int causal_off = sk - sq;  // key j visible to query i iff j <= i + causal_off
  int kv_end = sk;
  if (p.causal) kv_end = min(sk, q0 + BQ + causal_off);
  const int ntiles = (kv_end + BKV - 1) / BKV;

  load_tile<HD>(sQ, gq, p.ldq, q0, sq);
  if (ntiles > 0) {
    load_tile<HD>(sK, gk, p.ldk, 0, sk);
    load_tile<HD>(sV, gv, p.ldv, 0, sk);
  }
  cp_async_commit();

  constexpr int KS = HD / 16;  // k-steps of QK^T
  constexpr int NO = HD / 8;   // n-tiles of O
  uint32_t qf[KS][4];
  float o[NO][4];
#pragma unroll
  for (int i = 0; i < NO; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float mrow[2] = {-INFINITY, -INFINITY};
  float lrow[2] = {0.f, 0.f};
  const float sl2 = p.scale * 1.4426950408889634f;

  const int lm = lane >> 3, lr = lane & 7;  // ldmatrix: matrix index / row within matrix for this lane's address
  const int row_a = q0 + warp * 16 + (lane >> 2);  // query index (within sequence) of accumulator rows c0/c1
  const int row_b = row_a + 8;                     //   and c2/c3
  DropKey dk;
  unsigned long long e_a = 0, e_b = 0;             // dropout element index of (row_a, key 0) / (row_b, key 0)
  if constexpr (DROP) {
    dk = drop_key(p.drop);
    e_a = ((unsigned long long)(b * p.heads_q + h) * sq + row_a) * sk;
    e_b = e_a + 8ull * sk;
  }

  for (int t = 0; t < ntiles; ++t) {
    const int st = t & 1;
    if (t + 1 < ntiles) {
      load_tile<HD>(sK + (st ^ 1) * C::kTileBytes, gk, p.ldk, (t + 1) * BKV, sk);
      load_tile<HD>(sV + (st ^ 1) * C::kTileBytes, gv, p.ldv, (t + 1) * BKV, sk);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    if (t == 0) {
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t a = smem_u32(sQ + (warp * 16 + lr + (lm & 1) * 8) * C::kRowBytes + (ks * 16 + (lm >> 1) * 8) * 2);
        ldsm_x4(a, qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
      }
    }
    const uint8_t* cK = sK + st * C::kTileBytes;
    const uint8_t* cV = sV + st * C::kTileBytes;

    // ---- S = Q K^T  (16 x 64 per warp)
    float s[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
      for (int np = 0; np < 4; ++np) {  // pairs of 8-key n-tiles
        uint32_t b0, b1, b2, b3;
        const uint32_t a = smem_u32(cK + (np * 16 + (lm >> 1) * 8 + lr) * C::kRowBytes + (ks * 16 + (lm & 1) * 8) * 2);
        ldsm_x4(a, b0, b1, b2, b3);
        mma_bf16(s[2 * np], qf[ks], b0, b1);
        mma_bf16(s[2 * np + 1], qf[ks], b2, b3);
      }
    }
    // ---- mask + online softmax
    const int kbase = t * BKV + (lane & 3) * 2;
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = kbase + i * 8 + (e & 1);
        const int qi = (e < 2) ? row_a : row_b;
        bool vis = key < sk;
        if (p.causal) vis = vis && (key <= qi + causal_off);
        s[i][e] = vis ? s[i][e] * sl2 : -INFINITY;
        mx[e >> 1] = fmaxf(mx[e >> 1], s[i][e]);
      }
    }
    float corr[2], muse[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float mnew = fmaxf(mrow[r], mx[r]);
      muse[r] = (mnew == -INFINITY) ? 0.f : mnew;
      corr[r] = exp2f(mrow[r] - muse[r]);  // mrow = -inf on the first tile -> 0
      mrow[r] = mnew;
      lrow[r] *= corr[r];
    }
    float ls[2] = {0.f, 0.f};
    uint32_t pf[4][4];  // P as A-operand fragments: 4 k-steps of 16 keys
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float p0 = exp2f(s[i][0] - muse[0]), p1 = exp2f(s[i][1] - muse[0]);
      float p2 = exp2f(s[i][2] - muse[1]), p3 = exp2f(s[i][3] - muse[1]);
      ls[0] += p0 + p1;
      ls[1] += p2 + p3;
      if constexpr (DROP) {
        const float2 za = drop_mul2(dk, e_a + kbase + i * 8), zb = drop_mul2(dk, e_b + kbase + i * 8);
        p0 *= za.x, p1 *= za.y, p2 *= zb.x, p3 *= zb.y;
      }
      pf[i >> 1][(i & 1) * 2 + 0] = pack_bf16(p0, p1);
      pf[i >> 1][(i & 1) * 2 + 1] = pack_bf16(p2, p3);
    }
    lrow[0] += ls[0];
    lrow[1] += ls[1];
#pragma unroll
    for (int i = 0; i < NO; ++i) {
      o[i][0] *= corr[0], o[i][1] *= corr[0];
      o[i][2] *= corr[1], o[i][3] *= corr[1];
    }
    // ---- O += P V
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {  // 16 keys per step
#pragma unroll
      for (int np = 0; np < NO / 2; ++np) {  // pairs of 8-wide d n-tiles
        uint32_t b0, b1, b2, b3;
        const uint32_t a = smem_u32(cV + (kk * 16 + (lm & 1) * 8 + lr) * C::kRowBytes + (np * 16 + (lm >> 1) * 8) * 2);
        ldsm_x4_t(a, b0, b1, b2, b3);
        mma_bf16(o[2 * np], pf[kk], b0, b1);
        mma_bf16(o[2 * np + 1], pf[kk], b2, b3);
      }
    }
    __syncthreads();  // everyone done with stage st before it is refilled
  }
  cp_async_wait<0>();

  // ---- finalise: row sums across the quad, normalise, store
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    lrow[r] += __shfl_xor_sync(0xffffffffu, lrow[r], 1);
    lrow[r] += __shfl_xor_sync(0xffffffffu, lrow[r], 2);
  }
  const float inv0 = lrow[0] > 0.f ? 1.f / lrow[0] : 0.f;
  const float inv1 = lrow[1] > 0.f ? 1.f / lrow[1] : 0.f;
  bf16* go = p.o + (long)q_start * p.ldo + h * HD + (lane & 3) * 2;
#pragma unroll
  for (int i = 0; i < NO; ++i) {
    if (row_a < sq) *reinterpret_cast<uint32_t*>(go + (long)row_a * p.ldo + i * 8) = pack_bf16(o[i][0] * inv0, o[i][1] * inv0);
    if (row_b < sq) *reinterpret_cast<uint32_t*>(go + (long)row_b * p.ldo + i * 8) = pack_bf16(o[i][2] * inv1, o[i][3] * inv1);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Short-sequence kernel (head_dim 48, <= 8 heads, seq_q <= 32, seq_k <= 64): the NavDP decoder's self / cross attention,
// the Q-former self-attention and the goal compressor.  One CTA per query sequence, one warp per head.  Q, K, V rows
// (all heads, contiguous in memory) are staged with fully coalesced 16-byte cp.async; each warp runs QK^T, a
// single-pass softmax and PV for its head on mma.sync; O is staged back through the Q tile and written coalesced.
// The generic kernel above spent 4x the work on padding at these shapes (profiles/r1_ncu_small_v0_summary.txt).
template <int NKP, bool DROP>  // key tiles of 16; DROP: dropout on the probabilities, as in attn_kernel
__global__ void __launch_bounds__(256) attn_small_kernel(const AttnKParams<DROP> p, const int G) {
  constexpr int HD = 48;
  extern __shared__ __align__(16) uint8_t ssm[];
  const int heads = p.heads_q;
  const int RS = heads * HD * 2 + 16;  // row stride in bytes (+16: conflict-free ldmatrix)
  const int sq = p.seq_q, sk = p.seq_k;
  const int sq_pad = (sq + 15) & ~15;
  constexpr int sk_pad = NKP * 16;
  uint8_t* sQ = ssm;
  uint8_t* sK = sQ + sq_pad * RS;
  uint8_t* sV = sK + sk_pad * RS;
  // G consecutive query sequences that share one K/V sequence (G divides kv_div) are handled by one CTA: K/V is
  // staged once, Q / O tiles are cycled through the same buffer.
  const int b0 = blockIdx.x * G;
  const int kb = b0 / p.kv_div;
  const bf16* gk = p.k + (long)kb * sk * p.ldk;
  const bf16* gv = p.v + (long)kb * sk * p.ldv;
  const int chunks = heads * HD / 8;  // 16-byte chunks per row
  auto load_q = [&](int b) {
    const bf16* gq = p.q + (long)b * sq * p.ldq;
    for (int c = threadIdx.x; c < sq_pad * chunks; c += blockDim.x) {
      const int r = c / chunks, ch = c % chunks;
      cp_async16(sQ + r * RS + ch * 16, gq + (long)(r < sq ? r : 0) * p.ldq + ch * 8, r < sq);
    }
  };
  load_q(b0);
  for (int c = threadIdx.x; c < sk_pad * chunks; c += blockDim.x) {
    const int r = c / chunks, ch = c % chunks;
    const bool ok = r < sk;
    cp_async16(sK + r * RS + ch * 16, gk + (long)(ok ? r : 0) * p.ldk + ch * 8, ok);
    cp_async16(sV + r * RS + ch * 16, gv + (long)(ok ? r : 0) * p.ldv + ch * 8, ok);
  }
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();

  const int h = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int lm = lane >> 3, lr = lane & 7;
  const float sl2 = p.scale * 1.4426950408889634f;
  const int causal_off = sk - sq;
  for (int g = 0; g < G; ++g) {
  const int b = b0 + g;
  if (g > 0) {  // previous O tile has been written out (barrier at the end of the loop body): refill Q
    load_q(b);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
  }
  if (h < heads) {
    for (int mt = 0; mt < sq_pad / 16; ++mt) {
      uint32_t qf[3][4];
#pragma unroll
      for (int ks = 0; ks < 3; ++ks)
        ldsm_x4(smem_u32(sQ + (mt * 16 + lr + (lm & 1) * 8) * RS + h * 96 + (ks * 16 + (lm >> 1) * 8) * 2), qf[ks][0],
                qf[ks][1], qf[ks][2], qf[ks][3]);
      float s[2 * NKP][4];
#pragma unroll
      for (int i = 0; i < 2 * NKP; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 3; ++ks)
#pragma unroll
        for (int np = 0; np < NKP; ++np) {
          uint32_t b0, b1, b2, b3;
          ldsm_x4(smem_u32(sK + (np * 16 + (lm >> 1) * 8 + lr) * RS + h * 96 + (ks * 16 + (lm & 1) * 8) * 2), b0, b1, b2, b3);
          mma_bf16(s[2 * np], qf[ks], b0, b1);
          mma_bf16(s[2 * np + 1], qf[ks], b2, b3);
        }
      const int row_a = mt * 16 + (lane >> 2), row_b = row_a + 8;
      float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int i = 0; i < 2 * NKP; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = i * 8 + (lane & 3) * 2 + (e & 1);
          const int qi = e < 2 ? row_a : row_b;
          bool vis = key < sk;
          if (p.causal) vis = vis && key <= qi + causal_off;
          s[i][e] = vis ? s[i][e] * sl2 : -INFINITY;
          mx[e >> 1] = fmaxf(mx[e >> 1], s[i][e]);
        }
      float sum[2] = {0.f, 0.f};
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
        if (mx[r] == -INFINITY) mx[r] = 0.f;
      }
      uint32_t pf[NKP][4];
      DropKey dk;
      unsigned long long e_a = 0, e_b = 0;
      if constexpr (DROP) {
        dk = drop_key(p.drop);
        e_a = ((unsigned long long)(b * heads + h) * sq + row_a) * sk + (lane & 3) * 2;
        e_b = e_a + 8ull * sk;
      }
#pragma unroll
      for (int i = 0; i < 2 * NKP; ++i) {
        float p0 = exp2f(s[i][0] - mx[0]), p1 = exp2f(s[i][1] - mx[0]);
        float p2 = exp2f(s[i][2] - mx[1]), p3 = exp2f(s[i][3] - mx[1]);
        sum[0] += p0 + p1, sum[1] += p2 + p3;
        if constexpr (DROP) {
          const float2 za = drop_mul2(dk, e_a + i * 8), zb = drop_mul2(dk, e_b + i * 8);
          p0 *= za.x, p1 *= za.y, p2 *= zb.x, p3 *= zb.y;
        }
        pf[i >> 1][(i & 1) * 2 + 0] = pack_bf16(p0, p1);
        pf[i >> 1][(i & 1) * 2 + 1] = pack_bf16(p2, p3);
      }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 1);
        sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 2);
      }
      float o[6][4];
#pragma unroll
      for (int i = 0; i < 6; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < NKP; ++kk)
#pragma unroll
        for (int np = 0; np < 3; ++np) {
          uint32_t b0, b1, b2, b3;
          ldsm_x4_t(smem_u32(sV + (kk * 16 + (lm & 1) * 8 + lr) * RS + h * 96 + (np * 16 + (lm >> 1) * 8) * 2), b0, b1, b2, b3);
          mma_bf16(o[2 * np], pf[kk], b0, b1);
          mma_bf16(o[2 * np + 1], pf[kk], b2, b3);
        }
      const float inv0 = sum[0] > 0.f ? 1.f / sum[0] : 0.f, inv1 = sum[1] > 0.f ? 1.f / sum[1] : 0.f;
      // stage O over this warp's own (rows of this m-tile, head columns) slice of the Q tile: nobody else reads it
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        uint8_t* d = sQ + h * 96 + (i * 8 + (lane & 3) * 2) * 2;
        *reinterpret_cast<uint32_t*>(d + row_a * RS) = pack_bf16(o[i][0] * inv0, o[i][1] * inv0);
        *reinterpret_cast<uint32_t*>(d + row_b * RS) = pack_bf16(o[i][2] * inv1, o[i][3] * inv1);
      }
    }
  }
  __syncthreads();
  bf16* go = p.o + (long)b * sq * p.ldo;
  for (int c = threadIdx.x; c < sq * chunks; c += blockDim.x) {
    const int r = c / chunks, ch = c % chunks;
    *reinterpret_cast<uint4*>(go + (long)r * p.ldo + ch * 8) = *reinterpret_cast<const uint4*>(sQ + r * RS + ch * 16);
  }
  __syncthreads();  // O tile drained before the next sequence's Q overwrites it
  }  // g
}

template <int NKP, bool DROP = false>
void launch_attn_small(const AttnParams& p, cudaStream_t stream) {
  const int RS = p.heads_q * 96 + 16;
  const int smem = (((p.seq_q + 15) & ~15) + 2 * NKP * 16) * RS;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(attn_small_kernel<NKP, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (32 + 2 * NKP * 16) * (8 * 96 + 16));
    attr_set = true;
  }
  int G = 1;  // sequences per CTA: only when they share K/V
  if (p.kv_div % 4 == 0 && p.batch % 4 == 0) G = 4;
  else if (p.kv_div % 2 == 0 && p.batch % 2 == 0) G = 2;
  attn_small_kernel<NKP, DROP><<<p.batch / G, p.heads_q * 32, smem, stream>>>(p, G);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

template <int HD, bool DROP = false>
void launch_attn(const AttnParams& p, cudaStream_t stream) {
  using C = ACfg<HD>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(attn_kernel<HD, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    attr_set = true;
  }
  const int maxq = p.cu_q ? p.max_seq_q : p.seq_q;
  dim3 grid((maxq + BQ - 1) / BQ, p.heads_q, p.batch);
  attn_kernel<HD, DROP><<<grid, 128, C::kSmemBytes, stream>>>(p);
  prof_count_launch();
  N1_CUDA(cudaGetLastError());
}

}  // namespace

void attention(const AttnParams& p, cudaStream_t stream) {
  if (p.batch <= 0) return;
  N1_CHECK(p.heads_kv > 0 && p.heads_q % p.heads_kv == 0, "attention: heads_q must be a multiple of heads_kv");
  N1_CHECK(p.kv_div >= 1, "attention: kv_div >= 1");
  N1_CHECK(p.ldq % 8 == 0 && p.ldk % 8 == 0 && p.ldv % 8 == 0 && p.ldo % 2 == 0, "attention: misaligned strides");
  N1_CHECK(!p.cu_q || p.max_seq_q > 0, "attention: varlen needs max_seq_q");
  N1_CHECK(p.batch <= 65535 && p.heads_q <= 65535, "attention: grid too large");
  if (p.drop.rng) {  // training: the NavDP decoder / Q-former attention (8 heads x 48, fixed length)
    N1_CHECK(p.hd == 48 && !p.cu_q && !p.cu_k && !p.k_len && p.heads_q == p.heads_kv && p.kv_div == 1 && p.ldo % 8 == 0,
             "attention: dropout needs fixed-length multi-head attention with head_dim 48, kv_div 1");
    if (p.heads_q <= 8 && p.seq_q <= 32 && p.seq_k <= 64) {
      const int nkp = (p.seq_k + 15) / 16;
      if (nkp == 1) launch_attn_small<1, true>(p, stream);
      else if (nkp == 2) launch_attn_small<2, true>(p, stream);
      else if (nkp == 3) launch_attn_small<3, true>(p, stream);
      else launch_attn_small<4, true>(p, stream);
    } else {
      launch_attn<48, true>(p, stream);
    }
    return;
  }
  if (p.hd == 48 && !p.cu_q && !p.cu_k && !p.k_len && p.heads_q == p.heads_kv && p.heads_q <= 8 && p.seq_q <= 32 && p.seq_k <= 64 &&
      p.ldo % 8 == 0) {
    const int nkp = (p.seq_k + 15) / 16;
    if (nkp == 1) launch_attn_small<1>(p, stream);
    else if (nkp == 2) launch_attn_small<2>(p, stream);
    else if (nkp == 3) launch_attn_small<3>(p, stream);
    else launch_attn_small<4>(p, stream);
    return;
  }
  if (p.hd == 128 && attention_tc_supported(p)) {
    static int tc = -1;  // N1_ATTN_TC=0 keeps the mma.sync kernel
    if (tc < 0) {
      const char* e = getenv("N1_ATTN_TC");
      tc = e ? atoi(e) : 1;
    }
    if (tc) {
      attention_tc128(p, stream);
      return;
    }
  }
  switch (p.hd) {
    case 48: launch_attn<48>(p, stream); break;
    case 64: launch_attn<64>(p, stream); break;
    case 80: launch_attn<80>(p, stream); break;
    case 128: launch_attn<128>(p, stream); break;
    default: throw Error(-2, "attention: unsupported head_dim " + std::to_string(p.hd));
  }
}

}  // namespace n1
