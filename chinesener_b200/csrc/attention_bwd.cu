// Backward of the BERT self-attention core (sm_100a), head_dim 64, padded layout:
//   given qkv (bf16 [B*L, 3*NH*64]), the forward context O (bf16) and dO (bf16), produce
//   d_qkv (bf16, same layout as qkv).  This is the gradient tf.gradients derives through
//   attention_layer() of bert_base.bert.modeling (reference tools/train_utils.py:314).
//
// One CTA per (batch row, head).  Q, K, V and dO of the head are staged once in shared memory;
// nothing of size L x L is ever written anywhere: the scores are recomputed from Q/K with warp-level
// mma.sync.m16n8k16 (bf16 in, fp32 accumulate), flash-attention style, in two phases.
//   phase A (a warp owns 16 query rows):  row max / 1/sum / D = rowsum(dO*O), then
//           dS = P o (dO V^T - D),  dQ = scale * dS K                       (no cross-warp reduction)
//   phase B (a warp owns 16 key rows):    S^T = K Q^T so keys are the accumulator rows,
//           dV = P^T dO,  dK = scale * dS^T Q                               (no cross-warp reduction)
#include "common.cuh"

namespace {

using namespace nerdev;

constexpr int D = 64;
constexpr int PITCH = D + 8;  // bf16 per smem row (144 B): conflict-free fragment loads / ldmatrix
constexpr int NW = 8;         // warps per CTA

__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x2_trans(uint32_t& r0, uint32_t& r1, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(smem_u32(p)));
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t lds32(const __nv_bfloat16* p) { return *reinterpret_cast<const uint32_t*>(p); }

// A-operand fragments (16 rows x 64 k) of rows r0 / r1 = r0 + 8 of a [rows][PITCH] smem matrix
__device__ __forceinline__ void load_a_frags(uint32_t (&a)[4][4], const __nv_bfloat16* base, int r0, int cq) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    a[ks][0] = lds32(base + r0 * PITCH + ks * 16 + cq);
    a[ks][1] = lds32(base + (r0 + 8) * PITCH + ks * 16 + cq);
    a[ks][2] = lds32(base + r0 * PITCH + ks * 16 + 8 + cq);
    a[ks][3] = lds32(base + (r0 + 8) * PITCH + ks * 16 + 8 + cq);
  }
}
// acc[nt] (16 x 64 cols in 8 n-tiles) = A(16 x 64) · Bm^T where Bm is a [cols][PITCH] smem matrix (rows = n index)
__device__ __forceinline__ void mma_a_bt(float (&acc)[8][4], const uint32_t (&a)[4][4], const __nv_bfloat16* Bm, int n0,
                                         int lane, int cq) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const __nv_bfloat16* p = Bm + (n0 + nt * 8 + (lane >> 2)) * PITCH + ks * 16 + cq;
      mma16816(acc[nt], a[ks], lds32(p), lds32(p + 8));
    }
}
// out[dt] (16 x 64 dims) += P(16 x 64, C-fragment layout in p) · Bm[n0 .. n0+64][dims]
__device__ __forceinline__ void mma_p_b(float (&out)[8][4], const float (&p)[8][4], const __nv_bfloat16* Bm, int n0,
                                        int lane) {
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t pa[4];
    pa[0] = pack2(p[2 * kk][0], p[2 * kk][1]);
    pa[1] = pack2(p[2 * kk][2], p[2 * kk][3]);
    pa[2] = pack2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
    pa[3] = pack2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      uint32_t b0, b1;
      ldsm_x2_trans(b0, b1, Bm + (n0 + kk * 16 + (lane & 15)) * PITCH + dt * 8);
      mma16816(out[dt], pa, b0, b1);
    }
  }
}

// Same attention_probs dropout factor as the forward kernel (attention.cu): z in {0, 1/keep}.
// With O = (P o z) V:  dV = (P o z)^T dO,  dS = P o (z o dP - D),  D = rowsum(dO o O) unchanged.
__device__ __forceinline__ float attn_drop(uint32_t sa, uint32_t sb, int q, int k, uint32_t thr, float inv_keep) {
  return hash3(sa, (uint32_t)q, (uint32_t)k ^ sb) < thr ? inv_keep : 0.f;
}

template <bool DROP>
__global__ void __launch_bounds__(NW * 32)
bert_attention_bwd_kernel(const __nv_bfloat16* __restrict__ qkv, const int32_t* __restrict__ mask,
                          const __nv_bfloat16* __restrict__ ctx, const __nv_bfloat16* __restrict__ dctx,
                          __nv_bfloat16* __restrict__ dqkv, int Lpad, int NH, int Lp_max, float scale, float mask_add,
                          const int32_t* __restrict__ cu_seqlens, float keep, uint32_t seed_lo, uint32_t seed_hi) {
  const uint32_t dsa = seed_lo ^ ((uint32_t)(blockIdx.y * NH + blockIdx.x) * 0x9E3779B1u), dthr = keep_threshold(keep);
  const float dik = 1.f / keep;
  // padded mode: rows [b*L, (b+1)*L), keys masked by `mask`; packed mode: rows [cu[b], cu[b+1]), all keys valid and the
  // tile loops stop at the sequence's own length (same convention as the forward kernel, attention.cu)
  const size_t row_base = cu_seqlens ? (size_t)cu_seqlens[blockIdx.y] : (size_t)blockIdx.y * Lpad;
  const int L = cu_seqlens ? (cu_seqlens[blockIdx.y + 1] - cu_seqlens[blockIdx.y]) : Lpad;
  const int Lp = cu_seqlens ? (L + 63) / 64 * 64 : Lp_max;
  if (L == 0) return;
  extern __shared__ __align__(16) uint8_t smraw[];
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(smraw);
  __nv_bfloat16* Ks = Qs + (size_t)Lp * PITCH;
  __nv_bfloat16* Vs = Ks + (size_t)Lp * PITCH;
  __nv_bfloat16* Os = Vs + (size_t)Lp * PITCH;  // dO
  float* s_madd = reinterpret_cast<float*>(Os + (size_t)Lp * PITCH);
  float* s_m = s_madd + Lp;
  float* s_li = s_m + Lp;
  float* s_D = s_li + Lp;

  const int b = blockIdx.y, h = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int HD = NH * D;
  const size_t rs = (size_t)3 * HD;
  const __nv_bfloat16* base = qkv + row_base * rs + h * D;
  const __nv_bfloat16* obase = ctx + row_base * HD + h * D;
  const __nv_bfloat16* dobase = dctx + row_base * HD + h * D;

  for (int idx = tid; idx < Lp * 8; idx += NW * 32) {
    const int row = idx >> 3, ch = idx & 7;
    if (row < L) {
      cp_async16(Qs + row * PITCH + ch * 8, base + (size_t)row * rs + ch * 8);
      cp_async16(Ks + row * PITCH + ch * 8, base + (size_t)row * rs + HD + ch * 8);
      cp_async16(Vs + row * PITCH + ch * 8, base + (size_t)row * rs + 2 * HD + ch * 8);
      cp_async16(Os + row * PITCH + ch * 8, dobase + (size_t)row * HD + ch * 8);
    } else {
      const uint4 z = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(Qs + row * PITCH + ch * 8) = z;
      *reinterpret_cast<uint4*>(Ks + row * PITCH + ch * 8) = z;
      *reinterpret_cast<uint4*>(Vs + row * PITCH + ch * 8) = z;
      *reinterpret_cast<uint4*>(Os + row * PITCH + ch * 8) = z;
    }
  }
  cp_async_commit();
  for (int k = tid; k < Lp; k += NW * 32) {
    s_madd[k] = (k < L) ? (cu_seqlens ? 0.f : (1.f - (float)mask[(size_t)b * Lpad + k]) * mask_add) : -1e30f;
    s_m[k] = 0.f;
    s_li[k] = 0.f;
    s_D[k] = 0.f;
  }
  cp_async_wait<0>();
  __syncthreads();

  constexpr float kLog2e = 1.4426950408889634f;
  const int cq = 2 * (lane & 3);

  // ------------------------------------------------------------------ phase A: query rows
  for (int qb = warp; qb * 16 < L; qb += NW) {
    const int r0 = qb * 16 + (lane >> 2), r1 = r0 + 8;
    uint32_t qa[4][4], da[4][4];
    load_a_frags(qa, Qs, r0, cq);
    load_a_frags(da, Os, r0, cq);
    // D = rowsum(dO * O)
    float d0 = 0.f, d1 = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int col = ks * 16 + hh * 8 + cq;
        const __nv_bfloat162 g0 = *reinterpret_cast<const __nv_bfloat162*>(&da[ks][hh * 2 + 0]);
        const __nv_bfloat162 g1 = *reinterpret_cast<const __nv_bfloat162*>(&da[ks][hh * 2 + 1]);
        if (r0 < L) {
          const __nv_bfloat162 o = *reinterpret_cast<const __nv_bfloat162*>(obase + (size_t)r0 * HD + col);
          d0 += __low2float(g0) * __low2float(o) + __high2float(g0) * __high2float(o);
        }
        if (r1 < L) {
          const __nv_bfloat162 o = *reinterpret_cast<const __nv_bfloat162*>(obase + (size_t)r1 * HD + col);
          d1 += __low2float(g1) * __low2float(o) + __high2float(g1) * __high2float(o);
        }
      }
    d0 += __shfl_xor_sync(0xffffffffu, d0, 1);
    d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 1);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    // pass 1: row max and sum
    float m0 = -1e30f, m1 = -1e30f, l0 = 0.f, l1 = 0.f;
    for (int kb = 0; kb < Lp; kb += 64) {
      float s[8][4];
      mma_a_bt(s, qa, Ks, kb, lane, cq);
      float mx0 = -1e30f, mx1 = -1e30f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const float a0 = s_madd[kb + nt * 8 + cq], a1 = s_madd[kb + nt * 8 + cq + 1];
        s[nt][0] = s[nt][0] * scale + a0;
        s[nt][1] = s[nt][1] * scale + a1;
        s[nt][2] = s[nt][2] * scale + a0;
        s[nt][3] = s[nt][3] * scale + a1;
        mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float n0 = fmaxf(m0, mx0), n1 = fmaxf(m1, mx1);
      float p0 = 0.f, p1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        p0 += exp2f((s[nt][0] - n0) * kLog2e) + exp2f((s[nt][1] - n0) * kLog2e);
        p1 += exp2f((s[nt][2] - n1) * kLog2e) + exp2f((s[nt][3] - n1) * kLog2e);
      }
      l0 = l0 * exp2f((m0 - n0) * kLog2e) + p0;
      l1 = l1 * exp2f((m1 - n1) * kLog2e) + p1;
      m0 = n0;
      m1 = n1;
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float li0 = 1.f / l0, li1 = 1.f / l1;
    if ((lane & 3) == 0) {
      if (r0 < L) { s_m[r0] = m0; s_li[r0] = li0; s_D[r0] = d0; }
      if (r1 < L) { s_m[r1] = m1; s_li[r1] = li1; s_D[r1] = d1; }
    }
    // pass 2: dS and dQ
    float dq[8][4];
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) dq[dt][0] = dq[dt][1] = dq[dt][2] = dq[dt][3] = 0.f;
    for (int kb = 0; kb < Lp; kb += 64) {
      float s[8][4], dp[8][4];
      mma_a_bt(s, qa, Ks, kb, lane, cq);
      mma_a_bt(dp, da, Vs, kb, lane, cq);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const float a0 = s_madd[kb + nt * 8 + cq], a1 = s_madd[kb + nt * 8 + cq + 1];
        const float p00 = exp2f((s[nt][0] * scale + a0 - m0) * kLog2e) * li0;
        const float p01 = exp2f((s[nt][1] * scale + a1 - m0) * kLog2e) * li0;
        const float p10 = exp2f((s[nt][2] * scale + a0 - m1) * kLog2e) * li1;
        const float p11 = exp2f((s[nt][3] * scale + a1 - m1) * kLog2e) * li1;
        if (DROP) {
          const int k = kb + nt * 8 + cq;
          dp[nt][0] *= attn_drop(dsa, seed_hi, r0, k, dthr, dik);
          dp[nt][1] *= attn_drop(dsa, seed_hi, r0, k + 1, dthr, dik);
          dp[nt][2] *= attn_drop(dsa, seed_hi, r1, k, dthr, dik);
          dp[nt][3] *= attn_drop(dsa, seed_hi, r1, k + 1, dthr, dik);
        }
        s[nt][0] = p00 * (dp[nt][0] - d0);
        s[nt][1] = p01 * (dp[nt][1] - d0);
        s[nt][2] = p10 * (dp[nt][2] - d1);
        s[nt][3] = p11 * (dp[nt][3] - d1);
      }
      mma_p_b(dq, s, Ks, kb, lane);
    }
    __nv_bfloat16* dqb = dqkv + row_base * rs + h * D;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      if (r0 < L) *reinterpret_cast<uint32_t*>(dqb + (size_t)r0 * rs + dt * 8 + cq) = pack2(dq[dt][0] * scale, dq[dt][1] * scale);
      if (r1 < L) *reinterpret_cast<uint32_t*>(dqb + (size_t)r1 * rs + dt * 8 + cq) = pack2(dq[dt][2] * scale, dq[dt][3] * scale);
    }
  }
  __syncthreads();

  // ------------------------------------------------------------------ phase B: key rows
  for (int kb16 = warp; kb16 * 16 < L; kb16 += NW) {
    const int k0 = kb16 * 16 + (lane >> 2), k1 = k0 + 8;
    uint32_t ka[4][4], va[4][4];
    load_a_frags(ka, Ks, k0, cq);
    load_a_frags(va, Vs, k0, cq);
    const float ma0 = s_madd[k0], ma1 = s_madd[k1];
    float dk[8][4], dv[8][4];
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      dk[dt][0] = dk[dt][1] = dk[dt][2] = dk[dt][3] = 0.f;
      dv[dt][0] = dv[dt][1] = dv[dt][2] = dv[dt][3] = 0.f;
    }
    for (int qb = 0; qb < Lp; qb += 64) {
      float st[8][4], dpt[8][4];
      mma_a_bt(st, ka, Qs, qb, lane, cq);   // S^T  = K Q^T      (rows: keys, cols: queries)
      mma_a_bt(dpt, va, Os, qb, lane, cq);  // dP^T = V dO^T
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int q0 = qb + nt * 8 + cq, q1 = q0 + 1;
        const float mq0 = s_m[q0], mq1 = s_m[q1], lq0 = s_li[q0], lq1 = s_li[q1], dq0 = s_D[q0], dq1 = s_D[q1];
        const float p00 = exp2f((st[nt][0] * scale + ma0 - mq0) * kLog2e) * lq0;
        const float p01 = exp2f((st[nt][1] * scale + ma0 - mq1) * kLog2e) * lq1;
        const float p10 = exp2f((st[nt][2] * scale + ma1 - mq0) * kLog2e) * lq0;
        const float p11 = exp2f((st[nt][3] * scale + ma1 - mq1) * kLog2e) * lq1;
        float z00 = 1.f, z01 = 1.f, z10 = 1.f, z11 = 1.f;
        if (DROP) {
          z00 = attn_drop(dsa, seed_hi, q0, k0, dthr, dik);
          z01 = attn_drop(dsa, seed_hi, q1, k0, dthr, dik);
          z10 = attn_drop(dsa, seed_hi, q0, k1, dthr, dik);
          z11 = attn_drop(dsa, seed_hi, q1, k1, dthr, dik);
        }
        st[nt][0] = p00 * z00;
        st[nt][1] = p01 * z01;
        st[nt][2] = p10 * z10;
        st[nt][3] = p11 * z11;
        dpt[nt][0] = p00 * (z00 * dpt[nt][0] - dq0);
        dpt[nt][1] = p01 * (z01 * dpt[nt][1] - dq1);
        dpt[nt][2] = p10 * (z10 * dpt[nt][2] - dq0);
        dpt[nt][3] = p11 * (z11 * dpt[nt][3] - dq1);
      }
      mma_p_b(dv, st, Os, qb, lane);   // dV += P^T dO
      mma_p_b(dk, dpt, Qs, qb, lane);  // dK += dS^T Q
    }
    __nv_bfloat16* dkb = dqkv + row_base * rs + HD + h * D;
    __nv_bfloat16* dvb = dqkv + row_base * rs + 2 * HD + h * D;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      if (k0 < L) {
        *reinterpret_cast<uint32_t*>(dkb + (size_t)k0 * rs + dt * 8 + cq) = pack2(dk[dt][0] * scale, dk[dt][1] * scale);
        *reinterpret_cast<uint32_t*>(dvb + (size_t)k0 * rs + dt * 8 + cq) = pack2(dv[dt][0], dv[dt][1]);
      }
      if (k1 < L) {
        *reinterpret_cast<uint32_t*>(dkb + (size_t)k1 * rs + dt * 8 + cq) = pack2(dk[dt][2] * scale, dk[dt][3] * scale);
        *reinterpret_cast<uint32_t*>(dvb + (size_t)k1 * rs + dt * 8 + cq) = pack2(dv[dt][2], dv[dt][3]);
      }
    }
  }
}

}  // namespace

static int attention_bwd_launch(const void* qkv_bf16, const int32_t* mask, const void* ctx_bf16, const void* dctx_bf16,
                                void* dqkv_bf16, int B, int L, int num_heads, int head_dim, float scale, float mask_add,
                                const int32_t* cu_seqlens, float keep_prob, uint64_t seed, ner_stream_t stream) {
  if (B < 0 || L < 1 || num_heads < 1 || !(keep_prob > 0.f)) return NER_ERR_INVALID_ARG;
  if (B == 0) return NER_OK;
  if (!qkv_bf16 || (!mask && !cu_seqlens) || !ctx_bf16 || !dctx_bf16 || !dqkv_bf16) return NER_ERR_INVALID_ARG;
  if (head_dim != D) return NER_ERR_UNSUPPORTED;
  // Q/K/V and dO are staged with 16-byte cp.async copies, O is read and d_qkv written 4 bytes at a time
  if ((reinterpret_cast<uintptr_t>(qkv_bf16) & 15) != 0 || (reinterpret_cast<uintptr_t>(dctx_bf16) & 15) != 0 ||
      (reinterpret_cast<uintptr_t>(ctx_bf16) & 15) != 0 || (reinterpret_cast<uintptr_t>(dqkv_bf16) & 3) != 0)
    return NER_ERR_INVALID_ARG;
  const int Lp = (L + 63) / 64 * 64;
  const size_t smem = (size_t)4 * Lp * PITCH * 2 + (size_t)4 * Lp * 4;
  if (smem > 227 * 1024) return NER_ERR_UNSUPPORTED;  // L <= ~380
  auto kern = keep_prob < 1.f ? bert_attention_bwd_kernel<true> : bert_attention_bwd_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return NER_ERR_CUDA_BASE - (int)e;
  dim3 grid(num_heads, B);
  kern<<<grid, NW * 32, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(qkv_bf16), mask, static_cast<const __nv_bfloat16*>(ctx_bf16),
      static_cast<const __nv_bfloat16*>(dctx_bf16), static_cast<__nv_bfloat16*>(dqkv_bf16), L, num_heads, Lp, scale,
      mask_add, cu_seqlens, keep_prob, (uint32_t)seed, (uint32_t)(seed >> 32));
  return ner_launch_status();
}

extern "C" int ner_bert_attention_bwd(const void* qkv_bf16, const int32_t* mask, const void* ctx_bf16,
                                      const void* dctx_bf16, void* dqkv_bf16, int B, int L, int num_heads,
                                      int head_dim, float scale, float mask_add, float keep_prob, uint64_t seed,
                                      ner_stream_t stream) {
  if (!mask) return B == 0 ? NER_OK : NER_ERR_INVALID_ARG;
  return attention_bwd_launch(qkv_bf16, mask, ctx_bf16, dctx_bf16, dqkv_bf16, B, L, num_heads, head_dim, scale, mask_add,
                              nullptr, keep_prob, seed, stream);
}

extern "C" int ner_bert_attention_bwd_packed(const void* qkv_bf16, const int32_t* cu_seqlens, const void* ctx_bf16,
                                             const void* dctx_bf16, void* dqkv_bf16, int B, int L, int num_heads,
                                             int head_dim, float scale, float keep_prob, uint64_t seed,
                                             ner_stream_t stream) {
  if (!cu_seqlens) return B == 0 ? NER_OK : NER_ERR_INVALID_ARG;
  return attention_bwd_launch(qkv_bf16, nullptr, ctx_bf16, dctx_bf16, dqkv_bf16, B, L, num_heads, head_dim, scale, 0.f,
                              cu_seqlens, keep_prob, seed, stream);
}
