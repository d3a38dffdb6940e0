// Warp-level tensor-core attention over SHORT key sets (36 boxes, <= 128), bf16 in / fp32 accumulate.
//
//   sc_box_bias_all        BoxRelationalEmbedding + WG + ReLU + log for EVERY encoder layer in one pass
//                          (sparse_caption/models/relation_transformer.py:179-183,196-256).  The reference recomputes
//                          the [B,N,N,64] sin/cos embedding in each of the 6 layers; the embedding only depends on the
//                          boxes, so it is evaluated once per image pair and dotted with all L*h WG rows.
//   sc_bias_attention_fwd  box_attention (relation_transformer.py:258-293) given that bias:
//                          softmax(bias + mask(QK^T/sqrt(dk))) V, one WARP per (image, head).
//   cross-attention step   (sparse_caption/models/transformer.py:255-256,276,285-295) one warp per (image, head), the
//                          `beam` query rows of the image form the M dimension, so memory K/V are read once per image.
//
// The key sets are far too short for tcgen05 tiles (M=128/N>=8 with a TMEM round trip per 36x36 product); the products
// run on mma.sync.m16n8k16 straight out of shared memory (cp.async -> padded rows -> ldmatrix), scores and
// probabilities never leave registers.  These kernels are bound by the HBM bytes of Q,K,V,O (+ the bias tile).
#include "sc_common.cuh"

namespace {

constexpr int kDk = 64;               // head dim served by the mma path
constexpr int kPitch = (kDk + 8) * 2; // 144-byte rows: ldmatrix phases hit 8 distinct 16-byte bank groups

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *(uint32_t*)&t;
}

// rows [0, n) of a [*, 64] bf16 slice (row stride ld elements) -> smem rows of kPitch bytes.  Only the REAL rows are staged:
// the ldmatrix row addresses of the padding rows (up to the next multiple of 16) point at one shared all-zero row instead
// (36 boxes: 36 instead of 48 rows per tile -> a third more warps per SM for these latency-bound kernels).
__device__ __forceinline__ void stage_tile(const __nv_bfloat16* __restrict__ src, size_t ld, int n, unsigned char* dst, int lane) {
  for (int idx = lane; idx < n * 8; idx += 32) {
    const int r = idx >> 3, c = idx & 7;
    cp_async16(dst + r * kPitch + c * 16, src + (size_t)r * ld + c * 8);
  }
}

// One m-tile (16 query rows starting at m0) of softmax(bias + mask(Q K^T / 8)) V for one warp.
// sQ/sK/sV: this warp's staged tiles (nq / nk real rows); zrow: shared-memory address of a zeroed kPitch-byte row that stands in
// for the padding rows.  Result rows < nq are written back over the Q rows of the m-tile (bf16, kPitch rows).
template <int NT>
__device__ __forceinline__ void attn_mtile(unsigned char* sQ, const unsigned char* sK, const unsigned char* sV, int m0,
                                           int nq, int nk, const float* __restrict__ bias, int bias_ld,
                                           const float* __restrict__ key_mask, int lane, uint32_t zrow) {
  const int g = lane >> 2, t = lane & 3;
  const int r0 = m0 + g, r1 = r0 + 8;
  // ---- S = Q K^T, accumulated on top of the geometry bias: its loads (the only global reads of the m-tile) are requested
  // before the MMAs instead of between them and the softmax ----
  float s[2 * NT][4];
#pragma unroll
  for (int n = 0; n < 2 * NT; ++n) { s[n][0] = 0.f; s[n][1] = 0.f; s[n][2] = 0.f; s[n][3] = 0.f; }
  float bv[2 * NT][4];
  if (bias) {
    const bool vec2 = (bias_ld & 1) == 0 && (((uintptr_t)bias) & 7) == 0;
#pragma unroll
    for (int n = 0; n < 2 * NT; ++n) {
      const int col = n * 8 + 2 * t;
      bv[n][0] = bv[n][1] = bv[n][2] = bv[n][3] = 0.f;
      if (vec2 && col + 1 < nk) {
        if (r0 < nq) { const float2 b2 = *(const float2*)(bias + (size_t)r0 * bias_ld + col); bv[n][0] = b2.x; bv[n][1] = b2.y; }
        if (r1 < nq) { const float2 b2 = *(const float2*)(bias + (size_t)r1 * bias_ld + col); bv[n][2] = b2.x; bv[n][3] = b2.y; }
      } else {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          if (col + c < nk && r0 < nq) bv[n][c] = bias[(size_t)r0 * bias_ld + col + c];
          if (col + c < nk && r1 < nq) bv[n][2 + c] = bias[(size_t)r1 * bias_ld + col + c];
        }
      }
    }
  }
  const int qrow = m0 + (lane & 7) + ((lane >> 3) & 1) * 8;
  const uint32_t qbase = qrow < nq ? smem_u32(sQ) + (uint32_t)(qrow * kPitch + (lane >> 4) * 16) : zrow + (uint32_t)((lane >> 4) * 16);
  const int krow = (lane & 7) + (lane >> 4) * 8;  // + 16 np
  uint32_t kaddr[NT];
#pragma unroll
  for (int np = 0; np < NT; ++np)
    kaddr[np] = krow + 16 * np < nk ? smem_u32(sK) + (uint32_t)((krow + 16 * np) * kPitch + ((lane >> 3) & 1) * 16) : zrow + (uint32_t)(((lane >> 3) & 1) * 16);
#pragma unroll
  for (int ks = 0; ks < kDk / 16; ++ks) {
    uint32_t a[4];
    ldsm_x4(qbase + ks * 32, a);
#pragma unroll
    for (int np = 0; np < NT; ++np) {
      uint32_t b[4];
      ldsm_x4(kaddr[np] + ks * 32, b);
      mma_bf16(s[2 * np], a, b[0], b[1]);
      mma_bf16(s[2 * np + 1], a, b[2], b[3]);
    }
  }
  // ---- scale, mask, bias, softmax (rows g and g+8 of the tile; a row lives in the 4 lanes of a quad) ----
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int n = 0; n < 2 * NT; ++n) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int col = n * 8 + 2 * t + c;
      float v0 = s[n][c] * 0.125f, v1 = s[n][2 + c] * 0.125f;  // / sqrt(64)
      if (col < nk) {
        if (key_mask && key_mask[col] == 0.f) { v0 = -1e9f; v1 = -1e9f; }
        if (bias) { v0 += bv[n][c]; v1 += bv[n][2 + c]; }
      } else {
        v0 = -INFINITY; v1 = -INFINITY;
      }
      s[n][c] = v0; s[n][2 + c] = v1;
      mx0 = fmaxf(mx0, v0); mx1 = fmaxf(mx1, v1);
    }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
  for (int n = 0; n < 2 * NT; ++n) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const float p0 = __expf(s[n][c] - mx0), p1 = __expf(s[n][2 + c] - mx1);
      s[n][c] = p0; s[n][2 + c] = p1;
      sum0 += p0; sum1 += p1;
    }
  }
  sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
  sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
  const float inv0 = 1.f / sum0, inv1 = 1.f / sum1;
  // ---- O = P V ----
  float o[kDk / 8][4];
#pragma unroll
  for (int n = 0; n < kDk / 8; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
  const int vrow = (lane & 7) + ((lane >> 3) & 1) * 8;  // + 16 kk
#pragma unroll
  for (int kk = 0; kk < NT; ++kk) {
    uint32_t a[4];
    a[0] = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
    a[1] = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
    a[2] = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
    a[3] = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
    const uint32_t vaddr = vrow + 16 * kk < nk ? smem_u32(sV) + (uint32_t)((vrow + 16 * kk) * kPitch + (lane >> 4) * 16) : zrow + (uint32_t)((lane >> 4) * 16);
#pragma unroll
    for (int dp = 0; dp < kDk / 16; ++dp) {
      uint32_t b[4];
      ldsm_x4_trans(vaddr + dp * 32, b);
      mma_bf16(o[2 * dp], a, b[0], b[1]);
      mma_bf16(o[2 * dp + 1], a, b[2], b[3]);
    }
  }
  // ---- stage the output tile over this m-tile's Q rows (no longer needed) ----
  __syncwarp();
#pragma unroll
  for (int n = 0; n < kDk / 8; ++n) {
    if (r0 < nq) *(uint32_t*)(sQ + r0 * kPitch + (n * 8 + 2 * t) * 2) = pack_bf16(o[n][0] * inv0, o[n][1] * inv0);
    if (r1 < nq) *(uint32_t*)(sQ + r1 * kPitch + (n * 8 + 2 * t) * 2) = pack_bf16(o[n][2] * inv1, o[n][3] * inv1);
  }
}

// 16-byte coalesced copy of rows [0, n) of the staged output to global
__device__ __forceinline__ void store_rows(const unsigned char* sO, int n, __nv_bfloat16* __restrict__ dst, size_t ld, int lane) {
  for (int idx = lane; idx < n * 8; idx += 32) {
    const int r = idx >> 3, c = idx & 7;
    *(uint4*)(dst + (size_t)r * ld + c * 8) = *(const uint4*)(sO + r * kPitch + c * 16);
  }
}

struct EncAttnArgs {
  const __nv_bfloat16* q; const __nv_bfloat16* k; const __nv_bfloat16* v; int ldq, ldk, ldv;
  const float* bias;      // [B, h, N, N]
  const float* att_mask;  // [B, N] or nullptr
  __nv_bfloat16* out; int ldo;
  int B, N, h, warps;
};

template <int NT>
__global__ void __launch_bounds__(128) enc_attn_mma_kernel(const EncAttnArgs a) {
  extern __shared__ __align__(16) unsigned char smem_x[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * a.warps + warp;
  // smem: [zero row][warp 0: Q K V (N rows each)][warp 1: ...]
  if (threadIdx.x < kPitch / 16) *(uint4*)(smem_x + threadIdx.x * 16) = make_uint4(0u, 0u, 0u, 0u);
  sc::pdl_launch();
  sc::pdl_wait();
  const int N = a.N;
  const bool live = w < a.B * a.h;
  const int b = live ? w / a.h : 0, hh = live ? w - b * a.h : 0;
  unsigned char* sQ = smem_x + kPitch + (size_t)warp * 3 * N * kPitch;
  unsigned char* sK = sQ + N * kPitch;
  unsigned char* sV = sK + N * kPitch;
  const size_t row0 = (size_t)b * N;
  if (live) {
    stage_tile(a.q + row0 * a.ldq + hh * kDk, a.ldq, N, sQ, lane);
    stage_tile(a.k + row0 * a.ldk + hh * kDk, a.ldk, N, sK, lane);
    stage_tile(a.v + row0 * a.ldv + hh * kDk, a.ldv, N, sV, lane);
  }
  cp_async_wait_all();
  __syncthreads();  // (the zero row is shared by the CTA's warps)
  if (!live) return;
  const float* bias = a.bias + ((size_t)b * a.h + hh) * N * N;
  const float* km = a.att_mask ? a.att_mask + (size_t)b * N : nullptr;
  const uint32_t zrow = smem_u32(smem_x);
  for (int m0 = 0; m0 < N; m0 += 16) attn_mtile<NT>(sQ, sK, sV, m0, N, N, bias, N, km, lane, zrow);
  __syncwarp();
  store_rows(sQ, N, a.out + row0 * a.ldo + hh * kDk, a.ldo, lane);
}

struct CrossAttnArgs {
  const __nv_bfloat16* q; int ldq;
  const __nv_bfloat16* mk; const __nv_bfloat16* mv; int ldm;
  const float* att_mask;
  __nv_bfloat16* out; int ldo;
  int B, NB, N, h, warps;
};

template <int NT>
__global__ void __launch_bounds__(256) cross_attn_mma_kernel(const CrossAttnArgs a) {
  extern __shared__ __align__(16) unsigned char smem_x[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * a.warps + warp;
  // smem: [zero row][warp 0: Q (beam rows) K V (N rows each)][warp 1: ...]
  if (threadIdx.x < kPitch / 16) *(uint4*)(smem_x + threadIdx.x * 16) = make_uint4(0u, 0u, 0u, 0u);
  sc::pdl_launch();
  sc::pdl_wait();
  const int N = a.N;
  const bool live = w < a.B * a.h;
  const int b = live ? w / a.h : 0, hh = live ? w - b * a.h : 0;
  unsigned char* sQ = smem_x + kPitch + (size_t)warp * (2 * N + a.NB) * kPitch;
  unsigned char* sK = sQ + a.NB * kPitch;
  unsigned char* sV = sK + N * kPitch;
  if (live) {
    stage_tile(a.q + (size_t)b * a.NB * a.ldq + hh * kDk, a.ldq, a.NB, sQ, lane);
    stage_tile(a.mk + (size_t)b * N * a.ldm + hh * kDk, a.ldm, N, sK, lane);
    stage_tile(a.mv + (size_t)b * N * a.ldm + hh * kDk, a.ldm, N, sV, lane);
  }
  cp_async_wait_all();
  __syncthreads();  // (the zero row is shared by the CTA's warps)
  if (!live) return;
  const float* km = a.att_mask ? a.att_mask + (size_t)b * N : nullptr;
  attn_mtile<NT>(sQ, sK, sV, 0, a.NB, N, nullptr, 0, km, lane, smem_u32(smem_x));
  __syncwarp();
  store_rows(sQ, a.NB, a.out + (size_t)b * a.NB * a.ldo + hh * kDk, a.ldo, lane);
}

// 17 .. 32 beams: cross_attn_mma_kernel with a second query m-tile against the same staged K / V (a separate kernel so that
// the <= 16-beam kernel keeps its code).
template <int NT>
__global__ void __launch_bounds__(256) cross_attn_mma_wide_kernel(const CrossAttnArgs a) {
  extern __shared__ __align__(16) unsigned char smem_x[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * a.warps + warp;
  // smem: [zero row][warp 0: Q (beam rows) K V (N rows each)][warp 1: ...]
  if (threadIdx.x < kPitch / 16) *(uint4*)(smem_x + threadIdx.x * 16) = make_uint4(0u, 0u, 0u, 0u);
  sc::pdl_launch();
  sc::pdl_wait();
  const int N = a.N;
  const bool live = w < a.B * a.h;
  const int b = live ? w / a.h : 0, hh = live ? w - b * a.h : 0;
  unsigned char* sQ = smem_x + kPitch + (size_t)warp * (2 * N + a.NB) * kPitch;
  unsigned char* sK = sQ + a.NB * kPitch;
  unsigned char* sV = sK + N * kPitch;
  if (live) {
    stage_tile(a.q + (size_t)b * a.NB * a.ldq + hh * kDk, a.ldq, a.NB, sQ, lane);
    stage_tile(a.mk + (size_t)b * N * a.ldm + hh * kDk, a.ldm, N, sK, lane);
    stage_tile(a.mv + (size_t)b * N * a.ldm + hh * kDk, a.ldm, N, sV, lane);
  }
  cp_async_wait_all();
  __syncthreads();  // (the zero row is shared by the CTA's warps)
  if (!live) return;
  const float* km = a.att_mask ? a.att_mask + (size_t)b * N : nullptr;
  attn_mtile<NT>(sQ, sK, sV, 0, a.NB, N, nullptr, 0, km, lane, smem_u32(smem_x));
  attn_mtile<NT>(sQ, sK, sV, 16, a.NB, N, nullptr, 0, km, lane, smem_u32(smem_x));
  __syncwarp();
  store_rows(sQ, a.NB, a.out + (size_t)b * a.NB * a.ldo + hh * kDk, a.ldo, lane);
}

// ---- geometry bias for all layers: bias[l, b, hh, i, j] = log(max(relu(WG_{l,hh} . emb(i,j) + b_{l,hh}), 1e-6)) ----
struct DimMat8 { float v[8]; };

__global__ void __launch_bounds__(128) box_bias_all_kernel(const float* __restrict__ boxes, const float* __restrict__ wg_w,
                                                           const float* __restrict__ wg_b, float* __restrict__ bias,
                                                           int B, int N, int LH, int h, int trig, DimMat8 dm) {
  extern __shared__ __align__(16) float s_w[];  // [LH][dim_g] + [LH]
  const int dim_g = trig ? 64 : 4;
  for (int i = threadIdx.x; i < LH * dim_g; i += blockDim.x) s_w[i] = wg_w[i];
  for (int i = threadIdx.x; i < LH; i += blockDim.x) s_w[LH * dim_g + i] = wg_b[i];
  __syncthreads();
  const long pairs = (long)N * N;
  const long total = (long)B * pairs;
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const int b = (int)(p / pairs);
  const int r = (int)(p - (long)b * pairs);
  const int i = r / N, j = r - i * N;
  const float4 bi = *(const float4*)(boxes + ((size_t)b * N + i) * 4);
  const float4 bj = *(const float4*)(boxes + ((size_t)b * N + j) * 4);
  const float cxi = (bi.x + bi.z) * 0.5f, cyi = (bi.y + bi.w) * 0.5f, wi = (bi.z - bi.x) + 1.0f, hi = (bi.w - bi.y) + 1.0f;
  const float cxj = (bj.x + bj.z) * 0.5f, cyj = (bj.y + bj.w) * 0.5f, wj = (bj.z - bj.x) + 1.0f, hj = (bj.w - bj.y) + 1.0f;
  float delta[4];
  delta[0] = logf(fmaxf(fabsf((cxi - cxj) / wi), 1e-3f));
  delta[1] = logf(fmaxf(fabsf((cyi - cyj) / hi), 1e-3f));
  delta[2] = logf(wi / wj);
  delta[3] = logf(hi / hj);
  const int L = LH / h;
  if (trig) {
    float emb[64];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float p100 = 100.0f * delta[c];
#pragma unroll
      for (int f = 0; f < 8; ++f) sincosf(p100 * dm.v[f], &emb[c * 8 + f], &emb[32 + c * 8 + f]);
    }
    for (int l = 0; l < L; ++l) {
      for (int hh = 0; hh < h; ++hh) {
        const int lh = l * h + hh;
        const float4* wr = (const float4*)(s_w + lh * 64);
        // same summation order as the per-layer kernel: for (c,f): acc += sin*w[c*8+f] + cos*w[32+c*8+f]
        float acc = 0.f;
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4) {
          const float4 ws = wr[q4], wc = wr[8 + q4];
          acc += emb[4 * q4 + 0] * ws.x + emb[32 + 4 * q4 + 0] * wc.x;
          acc += emb[4 * q4 + 1] * ws.y + emb[32 + 4 * q4 + 1] * wc.y;
          acc += emb[4 * q4 + 2] * ws.z + emb[32 + 4 * q4 + 2] * wc.z;
          acc += emb[4 * q4 + 3] * ws.w + emb[32 + 4 * q4 + 3] * wc.w;
        }
        const float gg = fmaxf(acc + s_w[LH * 64 + lh], 0.f);
        bias[((((size_t)l * B + b) * h + hh) * N + i) * N + j] = logf(fmaxf(gg, 1e-6f));
      }
    }
  } else {
    for (int l = 0; l < L; ++l)
      for (int hh = 0; hh < h; ++hh) {
        const int lh = l * h + hh;
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) acc += delta[c] * s_w[lh * 4 + c];
        const float gg = fmaxf(acc + s_w[LH * 4 + lh], 0.f);
        bias[((((size_t)l * B + b) * h + hh) * N + i) * N + j] = logf(fmaxf(gg, 1e-6f));
      }
  }
}

// ---- the same bias on the tensor cores (bf16 inference path): D[16 pairs, LH] = emb[16, 64] . WG^T[64, LH] on mma.sync tiles ----
// The fp32 kernel above spends 3072 FFMAs + 768 shared-memory weight loads per box pair (1.07 ms for 2560 images: 14 % of an encoder
// pass).  Here a warp owns tiles of 16 consecutive pairs: every lane evaluates exactly the 16 sin/cos pairs its A fragments need
// (rows g / g + 8, frequencies 2t / 2t + 1 of each of the 4 deltas: no value is computed twice in the warp) and 4 x LH/8 x 3
// m16n8k16 MMAs replace the FFMA loop.  Both operands are split into bf16 hi + lo parts (x = hi + lo to 2^-17) and the product
// is hi.hi + lo.hi + hi.lo (fp32 accumulation): ~1e-5 absolute on the pre-activation, i.e. fp32-grade - the tensor cores buy
// speed here, not a precision trade.  The remaining approximations: sin / cos by two-term Cody-Waite reduction + MUFU (abs 1e-6),
// log by MUFU.LG2 (the exact kernel stays the fp32 verification / training path).  WG^T fragments (hi | lo) sit in shared memory
// in per-lane order (one conflict-free LDS.128 per (k-step, n-tile)).
__device__ __forceinline__ void fast_sincos(float x, float& sn, float& cs) {
  const float k = rintf(x * 0.15915494309189535f);
  float r = fmaf(-k, 6.2831854820251465f, x);   // 2 pi = 6.2831854820251465 - 1.7484556e-7
  r = fmaf(k, 1.7484556e-7f, r);
  sn = __sinf(r); cs = __cosf(r);
}
// (x0, x1) -> packed bf16 hi pair and packed bf16 residual pair
__device__ __forceinline__ void split_bf16(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h2 = __floats2bfloat162_rn(x0, x1);
  const float2 hf = __bfloat1622float2(h2);
  const __nv_bfloat162 l2 = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
  hi = *(const uint32_t*)&h2; lo = *(const uint32_t*)&l2;
}

template <int NT>  // NT = LH / 8 output tiles of 8 (layer, head) columns
__global__ void __launch_bounds__(128) box_bias_all_tc_kernel(const float* __restrict__ boxes, const float* __restrict__ wg_w,
                                                              const float* __restrict__ wg_b, float* __restrict__ bias,
                                                              int B, int N, int h, DimMat8 dm) {
  __shared__ uint4 s_b[4 * NT * 32];  // [ks][nt][lane]: {b0 hi, b1 hi, b0 lo, b1 lo}
  __shared__ float s_dm[8];
  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  // B fragment of WG^T (k x n) for m16n8k16: b0 = W[n = 8 nt + g][k = 16 ks + 2t, + 1], b1 = W[n][k + 8, + 9]
  for (int idx = threadIdx.x; idx < 4 * NT * 32; idx += blockDim.x) {
    const int ln = idx & 31, nt = (idx >> 5) % NT, ks = idx / (32 * NT);
    const float* w = wg_w + (size_t)(nt * 8 + (ln >> 2)) * 64 + ks * 16 + 2 * (ln & 3);
    uint4 o;
    split_bf16(w[0], w[1], o.x, o.z);
    split_bf16(w[8], w[9], o.y, o.w);
    s_b[idx] = o;
  }
  if (threadIdx.x < 8) s_dm[threadIdx.x] = dm.v[threadIdx.x];
  __syncthreads();
  float wb[NT][2];
  uint32_t lh_off[NT][2];  // byte offset of the (layer, head) plane of this lane's two columns of each n tile (image 0; host: < 2^32)
  const int pairs = N * N;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int lh = nt * 8 + 2 * t + e;
      wb[nt][e] = __ldg(wg_b + lh);
      lh_off[nt][e] = (uint32_t)((((size_t)(lh / h) * B * h + lh % h) * pairs) * sizeof(float));
    }
  const int total = B * pairs;  // (host: < 2^31)
  const int tiles = (total + 15) / 16;
  // a warp walks a CONTIGUOUS range of tiles: its boxes stay in L1 and (image, pair) advance without divisions
  const int warps_total = gridDim.x * (blockDim.x >> 5);
  const int per_warp = (tiles + warps_total - 1) / warps_total;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int tile0 = w * per_warp, tile1 = min(tile0 + per_warp, tiles);
  const float f0 = s_dm[2 * t], f1 = s_dm[2 * t + 1];
  const float inv_n = 1.0f / (float)N;
  int bb0 = tile0 < tiles ? (tile0 * 16) / pairs : 0;
  int rr0 = tile0 * 16 - bb0 * pairs;  // first pair of the tile inside image bb0
  for (int tile = tile0; tile < tile1; ++tile) {
    // A fragments (hi | lo) of rows g and g + 8: k-step ks covers the columns of deltas 2 ks, 2 ks + 1; ks < 2: sin, ks >= 2: cos
    uint32_t ah[4][4], al[4][4];
    bool ok[2];
    uint32_t out_r[2];  // byte offset of (image, head 0, pair) of the lane's two rows
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      int rr = rr0 + g + 8 * r, bb = bb0;
      if (rr >= pairs) { rr -= pairs; ++bb; }  // (a tile spans at most two images: pairs >= 16 is checked by the host)
      ok[r] = bb < B;
      if (!ok[r]) { bb = B - 1; }
      out_r[r] = (uint32_t)(((size_t)bb * h * pairs + rr) * sizeof(float));
      const int i = (int)(((float)rr + 0.5f) * inv_n);  // exact for rr < 2^22
      const int j = rr - i * N;
      // the quad's lane t evaluates delta[t] (one log + one division), the other three arrive by shuffle
      const float4 bi = __ldg((const float4*)(boxes + ((size_t)bb * N + i) * 4));
      const float4 bj = __ldg((const float4*)(boxes + ((size_t)bb * N + j) * 4));
      const bool xdir = (t & 1) == 0;  // t = 0: dx / w, 1: dy / h, 2: w / w, 3: h / h
      const float lo_i = xdir ? bi.x : bi.y, hi_i = xdir ? bi.z : bi.w, lo_j = xdir ? bj.x : bj.y, hi_j = xdir ? bj.z : bj.w;
      const float ci = (lo_i + hi_i) * 0.5f, cj = (lo_j + hi_j) * 0.5f, si = (hi_i - lo_i) + 1.0f, sj = (hi_j - lo_j) + 1.0f;
      const float mine = logf(t < 2 ? fmaxf(fabsf((ci - cj) / si), 1e-3f) : si / sj);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float p100 = 100.0f * __shfl_sync(0xffffffffu, mine, (lane & ~3) | c);
        float s0, c0, s1, c1;
        fast_sincos(p100 * f0, s0, c0);
        fast_sincos(p100 * f1, s1, c1);
        // delta c -> k-step c / 2 (sin) and 2 + c / 2 (cos); register r (+ 2 for the odd delta: columns + 8)
        split_bf16(s0, s1, ah[c >> 1][r + 2 * (c & 1)], al[c >> 1][r + 2 * (c & 1)]);
        split_bf16(c0, c1, ah[2 + (c >> 1)][r + 2 * (c & 1)], al[2 + (c >> 1)][r + 2 * (c & 1)]);
      }
    }
    rr0 += 16;
    if (rr0 >= pairs) { rr0 -= pairs; ++bb0; }
    float d[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) { d[nt][0] = 0.f; d[nt][1] = 0.f; d[nt][2] = 0.f; d[nt][3] = 0.f; }
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint4 bw[NT];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) bw[nt] = s_b[(ks * NT + nt) * 32 + lane];
      // small terms first; consecutive MMAs go to different accumulators
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) mma_bf16(d[nt], al[ks], bw[nt].x, bw[nt].y);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) mma_bf16(d[nt], ah[ks], bw[nt].z, bw[nt].w);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) mma_bf16(d[nt], ah[ks], bw[nt].x, bw[nt].y);
    }
    // D: (row g, cols 2t, 2t+1), (row g + 8, cols 2t, 2t+1) of each n tile; column = layer * h + head
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = e >> 1;
        if (ok[r]) {  // log(max(relu(x), 1e-6)); the argument is never denormal: plain MUFU.LG2
          float l2;
          asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(fmaxf(d[nt][e] + wb[nt][e & 1], 1e-6f)));
          *(float*)((char*)bias + (out_r[r] + lh_off[nt][e & 1])) = l2 * 0.6931471805599453f;
        }
      }
  }
}

}  // namespace

extern "C" {

int sc_box_bias_all(const float* boxes, const float* wg_w, const float* wg_b, float* bias, int B, int N, int layers, int h,
                    int trig, float wave_len, cudaStream_t stream) {
  SC_CHECK(B > 0 && N > 0 && layers >= 1 && h >= 1, SC_ERR_SHAPE, "sc_box_bias_all: B=%d N=%d layers=%d h=%d", B, N, layers, h);
  SC_CHECK(((uintptr_t)boxes & 15) == 0 && ((uintptr_t)wg_w & 15) == 0, SC_ERR_ALIGN, "sc_box_bias_all: boxes / wg_w must be 16-byte aligned");
  const int LH = layers * h;
  const int dim_g = trig ? 64 : 4;
  const size_t smem = sizeof(float) * ((size_t)LH * dim_g + LH);
  SC_CHECK(smem <= 200 * 1024, SC_ERR_UNSUPPORTED, "sc_box_bias_all: %d WG rows do not fit in shared memory", LH);
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(box_bias_all_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr = true;
  }
  DimMat8 dm;
  for (int f = 0; f < 8; ++f) dm.v[f] = 1.0f / powf(wave_len, (float)f / 8.0f);
  const long total = (long)B * N * N;
  box_bias_all_kernel<<<(unsigned)((total + 127) / 128), 128, smem, stream>>>(boxes, wg_w, wg_b, bias, B, N, LH, h, trig, dm);
  SC_LAUNCH_CHECK("sc_box_bias_all");
  return SC_OK;
}

int sc_box_bias_all_tc(const float* boxes, const float* wg_w, const float* wg_b, float* bias, int B, int N, int layers, int h,
                       float wave_len, cudaStream_t stream) {
  SC_CHECK(B > 0 && N > 0 && layers >= 1 && h >= 1, SC_ERR_SHAPE, "sc_box_bias_all_tc: B=%d N=%d layers=%d h=%d", B, N, layers, h);
  SC_CHECK(((uintptr_t)boxes & 15) == 0, SC_ERR_ALIGN, "sc_box_bias_all_tc: boxes must be 16-byte aligned");
  const int LH = layers * h;
  SC_CHECK(LH % 8 == 0 && LH <= 64, SC_ERR_UNSUPPORTED, "sc_box_bias_all_tc: layers * h = %d must be a multiple of 8, at most 64 (use sc_box_bias_all)", LH);
  SC_CHECK(N >= 4 && N <= 2048 && (long)B * N * N < (1L << 31) - 16, SC_ERR_UNSUPPORTED,
           "sc_box_bias_all_tc: N=%d in [4, 2048] and B*N*N < 2^31 (use sc_box_bias_all)", N);
  SC_CHECK((size_t)LH * B * N * N * sizeof(float) < ((size_t)1 << 32), SC_ERR_UNSUPPORTED,
           "sc_box_bias_all_tc: the bias tensor must stay below 4 GB (32-bit byte offsets; use sc_box_bias_all or split the batch)");
  DimMat8 dm;
  for (int f = 0; f < 8; ++f) dm.v[f] = 1.0f / powf(wave_len, (float)f / 8.0f);
  const long tiles = ((long)B * N * N + 15) / 16;
  int sms = 148;
  { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); }
  long blocks = (tiles + 3) / 4;
  if (blocks > (long)sms * 8) blocks = (long)sms * 8;
#define TC_CASE(NTV) case NTV: box_bias_all_tc_kernel<NTV><<<(unsigned)blocks, 128, 0, stream>>>(boxes, wg_w, wg_b, bias, B, N, h, dm); break
  switch (LH / 8) {
    TC_CASE(1); TC_CASE(2); TC_CASE(3); TC_CASE(4); TC_CASE(5); TC_CASE(6); TC_CASE(7); TC_CASE(8);
    default: SC_CHECK(false, SC_ERR_UNSUPPORTED, "sc_box_bias_all_tc: LH=%d", LH);
  }
#undef TC_CASE
  SC_LAUNCH_CHECK("sc_box_bias_all_tc");
  return SC_OK;
}

int sc_bias_attention_fwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype, const float* bias,
                          const float* att_mask, void* out, int ldo, int B, int N, int h, int dk, cudaStream_t stream) {
  SC_CHECK(B > 0 && N > 0 && h > 0, SC_ERR_SHAPE, "sc_bias_attention_fwd: B=%d N=%d h=%d", B, N, h);
  SC_CHECK(dtype == SC_BF16, SC_ERR_DTYPE, "sc_bias_attention_fwd: bf16 only (fp32 runs sc_box_attention_fwd)");
  SC_CHECK(dk == kDk, SC_ERR_UNSUPPORTED, "sc_bias_attention_fwd: d_k=%d (tensor path serves d_k=64)", dk);
  SC_CHECK(N <= 128, SC_ERR_UNSUPPORTED, "sc_bias_attention_fwd: N=%d > 128", N);
  SC_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0, SC_ERR_ALIGN, "sc_bias_attention_fwd: ld %% 8");
  SC_CHECK((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) == 0, SC_ERR_ALIGN, "sc_bias_attention_fwd: 16-byte alignment");
  SC_CHECK(bias != nullptr, SC_ERR_SHAPE, "sc_bias_attention_fwd: bias missing");
  EncAttnArgs a;
  a.q = (const __nv_bfloat16*)q; a.k = (const __nv_bfloat16*)k; a.v = (const __nv_bfloat16*)v;
  a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.bias = bias; a.att_mask = att_mask; a.out = (__nv_bfloat16*)out; a.ldo = ldo;
  a.B = B; a.N = N; a.h = h;
  const int NT = (N + 15) / 16;
  const size_t per_warp = (size_t)3 * N * kPitch;  // only the real rows are staged (see stage_tile)
  int warps = (int)((200 * 1024 - kPitch) / per_warp);
  if (warps > 4) warps = 4;
  SC_CHECK(warps >= 1, SC_ERR_UNSUPPORTED, "sc_bias_attention_fwd: N=%d does not fit in shared memory", N);
  a.warps = warps;
  const size_t smem = per_warp * warps + kPitch;
  const int blocks = (B * h + warps - 1) / warps;
#define ENC_CASE(NTV)                                                                                              \
  case NTV: {                                                                                                      \
    static bool attr = false;                                                                                      \
    if (!attr) {                                                                                                   \
      cudaFuncSetAttribute(enc_attn_mma_kernel<NTV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);     \
      attr = true;                                                                                                 \
    }                                                                                                              \
    sc::launch_pdl(enc_attn_mma_kernel<NTV>, dim3(blocks), dim3(32 * warps), smem, stream, a);                     \
  } break
  switch (NT) {
    ENC_CASE(1); ENC_CASE(2); ENC_CASE(3); ENC_CASE(4); ENC_CASE(5); ENC_CASE(6); ENC_CASE(7); ENC_CASE(8);
    default: SC_CHECK(false, SC_ERR_UNSUPPORTED, "sc_bias_attention_fwd: N=%d", N);
  }
#undef ENC_CASE
  SC_LAUNCH_CHECK("sc_bias_attention_fwd");
  return SC_OK;
}

}  // extern "C"

// bf16, d_k = 64 cross-attention step on the tensor path; returns SC_ERR_UNSUPPORTED when the shape is not served
// (sc_decode_cross_attn_step in sc_decode.cu then runs its generic kernel).
int sc_cross_attn_mma_launch(const void* q, int ldq, const void* mem_k, const void* mem_v, int ldm, const float* att_mask,
                             void* out, int ldo, int B, int beam, int N, int h, cudaStream_t stream) {
  if (beam > 32 || N > 128) return SC_ERR_UNSUPPORTED;
  if ((((uintptr_t)q | (uintptr_t)mem_k | (uintptr_t)mem_v | (uintptr_t)out) & 15) != 0) return SC_ERR_UNSUPPORTED;
  CrossAttnArgs a;
  a.q = (const __nv_bfloat16*)q; a.ldq = ldq; a.mk = (const __nv_bfloat16*)mem_k; a.mv = (const __nv_bfloat16*)mem_v; a.ldm = ldm;
  a.att_mask = att_mask; a.out = (__nv_bfloat16*)out; a.ldo = ldo; a.B = B; a.NB = beam; a.N = N; a.h = h;
  const int NT = (N + 15) / 16;
  const size_t per_warp = (size_t)(2 * N + beam) * kPitch;  // only the real rows are staged (see stage_tile)
  // 6 warps x 10.8 KB (36 boxes, beam 3): three CTAs = 18 warps per SM keep ~170 KB of K / V requests in flight
  int warps = (int)((72 * 1024 - kPitch) / per_warp);
  if (warps > 8) warps = 8;
  if (warps < 1) return SC_ERR_UNSUPPORTED;
  a.warps = warps;
  const size_t smem = per_warp * warps + kPitch;
  const int blocks = (B * h + warps - 1) / warps;
#define X_CASE(KERN, NTV)                                                                                          \
  case NTV: {                                                                                                      \
    static bool attr = false;                                                                                      \
    if (!attr) {                                                                                                   \
      cudaFuncSetAttribute(KERN<NTV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);                    \
      attr = true;                                                                                                 \
    }                                                                                                              \
    sc::launch_pdl(KERN<NTV>, dim3(blocks), dim3(32 * warps), smem, stream, a);                                    \
  } break
#define X_CASES(KERN)                                                                                              \
  switch (NT) {                                                                                                    \
    X_CASE(KERN, 1); X_CASE(KERN, 2); X_CASE(KERN, 3); X_CASE(KERN, 4);                                            \
    X_CASE(KERN, 5); X_CASE(KERN, 6); X_CASE(KERN, 7); X_CASE(KERN, 8);                                            \
    default: return SC_ERR_UNSUPPORTED;                                                                            \
  }
  if (beam > 16) { X_CASES(cross_attn_mma_wide_kernel) }
  else { X_CASES(cross_attn_mma_kernel) }
#undef X_CASES
#undef X_CASE
  SC_LAUNCH_CHECK("sc_decode_cross_attn_step");
  return SC_OK;
}
