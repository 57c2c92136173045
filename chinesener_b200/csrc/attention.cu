// BERT self-attention core for sm_100a:  ctx = softmax(Q K^T * scale + (1-mask)*mask_add) V
// per (batch, head), head_dim = 64.  Replaces attention_layer() of bert_base.bert.modeling as
// executed from reference tools/layer.py:68-77 (semantics: SURVEY.md Appendix A.3).
//
// v1 uses warp-level mma.sync.m16n8k16 (bf16 in, fp32 accumulate) in a flash-style
// single pass: one CTA = 64 query rows of one (b, h); K and V of that head are staged once in
// shared memory with cp.async (row pitch 144 B -> conflict-free fragment loads / ldmatrix),
// scores and probabilities never leave registers.  (Attention is 2.7 % of the encoder FLOPs;
// the dense layers run on tcgen05 — see gemm_tc.cu.)
#include <stdlib.h>

#include "common.cuh"

namespace {

using namespace nerdev;

constexpr int D = 64;
constexpr int PITCH = D + 8;  // bf16 elements per smem row (144 B)
constexpr int QT = 64;        // query rows per CTA
constexpr int KB = 64;        // keys per inner block

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t& r0, uint32_t& r1, const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];"
               : "=r"(r0), "=r"(r1)
               : "r"(smem_u32(smem_row)));
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// attention_probs dropout (training): z(b,h,q,k) in {0, 1/keep} from the shared counter hash; the
// row sums keep the undropped probabilities (dropout follows the softmax in attention_layer()).
__device__ __forceinline__ float attn_drop(uint32_t sa, uint32_t sb, int q, int k, uint32_t thr, float inv_keep) {
  return hash3(sa, (uint32_t)q, (uint32_t)k ^ sb) < thr ? inv_keep : 0.f;
}

template <bool DROP>
__global__ void __launch_bounds__(128)
bert_attention_kernel(const __nv_bfloat16* __restrict__ qkv, const int32_t* __restrict__ mask,
                      __nv_bfloat16* __restrict__ ctx, int Lpad, int NH, int Lp_max, float scale, float mask_add,
                      const int32_t* __restrict__ cu_seqlens, float keep, uint32_t seed_lo, uint32_t seed_hi) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __align__(16) uint8_t smem_raw[];
  __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(smem_raw);
  __nv_bfloat16* Vs = Ks + (size_t)Lp_max * PITCH;
  float* s_madd = reinterpret_cast<float*>(Vs + (size_t)Lp_max * PITCH);

  const int b = blockIdx.z, h = blockIdx.y, qt = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int HD = NH * D;
  const size_t rs = (size_t)3 * HD;  // qkv row stride (elements)
  // padded mode: rows [b*L, (b+1)*L), keys masked by `mask`; packed mode: rows [cu[b], cu[b+1]), all valid
  const size_t row_base = cu_seqlens ? (size_t)cu_seqlens[b] : (size_t)b * Lpad;
  const int L = cu_seqlens ? (cu_seqlens[b + 1] - cu_seqlens[b]) : Lpad;
  if (qt * QT >= L) return;  // (whole CTA) nothing to do for this query tile
  const int Lp = cu_seqlens ? (L + KB - 1) / KB * KB : Lp_max;
  const __nv_bfloat16* base = qkv + row_base * rs;

  for (int idx = tid; idx < Lp * 8; idx += 128) {
    const int row = idx >> 3, ch = idx & 7;
    __nv_bfloat16* kd = Ks + row * PITCH + ch * 8;
    __nv_bfloat16* vd = Vs + row * PITCH + ch * 8;
    if (row < L) {
      const __nv_bfloat16* src = base + (size_t)row * rs + h * D + ch * 8;
      cp_async16(kd, src + HD);
      cp_async16(vd, src + 2 * HD);
    } else {
      *reinterpret_cast<uint4*>(kd) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(vd) = make_uint4(0, 0, 0, 0);
    }
  }
  cp_async_commit();
  for (int k = tid; k < Lp; k += 128)
    s_madd[k] = (k < L) ? (cu_seqlens ? 0.f : (1.f - (float)mask[(size_t)b * Lpad + k]) * mask_add) : -1e30f;

  // Q fragments straight from global (each element read once)
  const int q0 = qt * QT + warp * 16;
  const int r0 = q0 + (lane >> 2), r1 = r0 + 8;
  const int cq = 2 * (lane & 3);
  uint32_t qa[4][4];
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    const __nv_bfloat16* p0 = base + (size_t)r0 * rs + h * D + ks * 16 + cq;
    const __nv_bfloat16* p1 = base + (size_t)r1 * rs + h * D + ks * 16 + cq;
    qa[ks][0] = (r0 < L) ? *reinterpret_cast<const uint32_t*>(p0) : 0u;
    qa[ks][1] = (r1 < L) ? *reinterpret_cast<const uint32_t*>(p1) : 0u;
    qa[ks][2] = (r0 < L) ? *reinterpret_cast<const uint32_t*>(p0 + 8) : 0u;
    qa[ks][3] = (r1 < L) ? *reinterpret_cast<const uint32_t*>(p1 + 8) : 0u;
  }
  cp_async_wait<0>();
  __syncthreads();

  constexpr float kLog2e = 1.4426950408889634f;
  float o[8][4];
#pragma unroll
  for (int dt = 0; dt < 8; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
  float m0 = -1e30f, m1 = -1e30f, l0 = 0.f, l1 = 0.f;

  if (q0 < L) {
    for (int kb = 0; kb < Lp; kb += KB) {
      float s[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const __nv_bfloat16* kp = Ks + (kb + nt * 8 + (lane >> 2)) * PITCH + ks * 16 + cq;
          const uint32_t b0 = *reinterpret_cast<const uint32_t*>(kp);
          const uint32_t b1 = *reinterpret_cast<const uint32_t*>(kp + 8);
          mma_bf16_16816(s[nt], qa[ks], b0, b1);
        }
      }
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
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
      const float c0 = exp2f((m0 - mn0) * kLog2e), c1 = exp2f((m1 - mn1) * kLog2e);
      m0 = mn0;
      m1 = mn1;
      float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = exp2f((s[nt][0] - mn0) * kLog2e);
        s[nt][1] = exp2f((s[nt][1] - mn0) * kLog2e);
        s[nt][2] = exp2f((s[nt][2] - mn1) * kLog2e);
        s[nt][3] = exp2f((s[nt][3] - mn1) * kLog2e);
        ps0 += s[nt][0] + s[nt][1];
        ps1 += s[nt][2] + s[nt][3];
      }
      l0 = l0 * c0 + ps0;
      l1 = l1 * c1 + ps1;
      if (DROP) {
        const uint32_t sa = seed_lo ^ ((uint32_t)(b * NH + h) * 0x9E3779B1u), thr = keep_threshold(keep);
        const float ik = 1.f / keep;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int k = kb + nt * 8 + cq;
          s[nt][0] *= attn_drop(sa, seed_hi, r0, k, thr, ik);
          s[nt][1] *= attn_drop(sa, seed_hi, r0, k + 1, thr, ik);
          s[nt][2] *= attn_drop(sa, seed_hi, r1, k, thr, ik);
          s[nt][3] *= attn_drop(sa, seed_hi, r1, k + 1, thr, ik);
        }
      }
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) {
        o[dt][0] *= c0;
        o[dt][1] *= c0;
        o[dt][2] *= c1;
        o[dt][3] *= c1;
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t pa[4];
        pa[0] = pack2(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack2(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int dt = 0; dt < 8; ++dt) {
          uint32_t b0, b1;
          ldmatrix_x2_trans(b0, b1, Vs + (kb + kk * 16 + (lane & 15)) * PITCH + dt * 8);
          mma_bf16_16816(o[dt], pa, b0, b1);
        }
      }
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    __nv_bfloat16* ob = ctx + row_base * HD + h * D;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      if (r0 < L) *reinterpret_cast<uint32_t*>(ob + (size_t)r0 * HD + dt * 8 + cq) = pack2(o[dt][0] * inv0, o[dt][1] * inv0);
      if (r1 < L) *reinterpret_cast<uint32_t*>(ob + (size_t)r1 * HD + dt * 8 + cq) = pack2(o[dt][2] * inv1, o[dt][3] * inv1);
    }
  }
}

}  // namespace

int ner_bert_attention_tc(const void* qkv_bf16, const int32_t* mask, void* ctx_bf16, int B, int L, int num_heads, int head_dim,
                          float scale, float mask_add, const int32_t* cu_seqlens, int n_rows, cudaStream_t st);

static int attn_variant() {
  const char* e = getenv("NER_ATTN_VARIANT");   // tuning / test hook, read per call: 1 = mma.sync kernel everywhere
  return e ? atoi(e) : 0;
}

extern "C" int ner_bert_attention(const void* qkv_bf16, const int32_t* mask, void* ctx_bf16, int B, int L,
                                  int num_heads, int head_dim, float scale, float mask_add,
                                  const int32_t* cu_seqlens, int n_rows, float keep_prob, uint64_t seed,
                                  ner_stream_t stream) {
  if (B < 0 || L < 1 || num_heads < 1 || !(keep_prob > 0.f)) return NER_ERR_INVALID_ARG;
  if (B == 0) return NER_OK;
  if (!qkv_bf16 || (!mask && !cu_seqlens) || !ctx_bf16) return NER_ERR_INVALID_ARG;
  if (n_rows < 0 || (!cu_seqlens && n_rows != 0 && n_rows != B * L)) return NER_ERR_INVALID_ARG;
  if (head_dim != D) return NER_ERR_UNSUPPORTED;
  if (keep_prob >= 1.f && attn_variant() != 1) {
    // inference: tcgen05 kernel (S and O in tensor memory, operands by TMA); packed mode needs the row count of qkv
    const int rows = cu_seqlens ? n_rows : B * L;
    if (rows > 0) {
      const int rc = ner_bert_attention_tc(qkv_bf16, mask, ctx_bf16, B, L, num_heads, head_dim, scale, mask_add, cu_seqlens,
                                           rows, static_cast<cudaStream_t>(stream));
      if (rc != NER_ERR_UNSUPPORTED) return rc;
    }
  }
  // the K/V staging issues 16-byte cp.async copies (row stride 3*NH*64 bf16 keeps every row 16-byte aligned if the base is)
  if ((reinterpret_cast<uintptr_t>(qkv_bf16) & 15) != 0 || (reinterpret_cast<uintptr_t>(ctx_bf16) & 15) != 0)
    return NER_ERR_INVALID_ARG;
  const int Lp = (L + KB - 1) / KB * KB;
  const size_t smem = (size_t)2 * Lp * PITCH * 2 + (size_t)Lp * 4;
  if (smem > 227 * 1024) return NER_ERR_UNSUPPORTED;  // L <= ~780
  auto kern = keep_prob < 1.f ? bert_attention_kernel<true> : bert_attention_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return NER_ERR_CUDA_BASE - (int)e;
  dim3 grid((L + QT - 1) / QT, num_heads, B);
  e = ner_launch_pdl(kern, grid, dim3(128), smem, static_cast<cudaStream_t>(stream), static_cast<const __nv_bfloat16*>(qkv_bf16),
                     mask, static_cast<__nv_bfloat16*>(ctx_bf16), L, num_heads, Lp, scale, mask_add, cu_seqlens, keep_prob,
                     (uint32_t)seed, (uint32_t)(seed >> 32));
  if (e != cudaSuccess) return NER_ERR_CUDA_BASE - (int)e;
  return ner_launch_status();
}
