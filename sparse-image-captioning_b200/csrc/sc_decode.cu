// Incremental decoding kernels (K5, K6, K7, K8).
// Reference behaviour:
//   K5 self-attention step with growing cache  : sparse_caption/models/transformer.py:230-295 (cat(cache,k), softmax, PV)
//   K6 cross-attention step, cache re-use       : transformer.py:255-256,276
//   K7 beam step + finished-beam bookkeeping    : sparse_caption/models/caption_model.py:56-111,151-226
//      greedy step                              : transformer.py:507-561
//   K8 state reorder state[i][:, state_ix]      : caption_model.py:106-110
//
// Layout: rows r = image*beam + slot.  Self K/V caches are [slot s][row][D], written once and never moved; a
// beam's history is found through the ancestor table anc[row][s] (row that wrote slot s for this beam), which
// K7 rewrites each step (a [R,L] int gather) instead of gathering 24 cache tensors like the reference does.
// Cross K/V are per IMAGE ([B*N, D]) and shared by the beams of that image.
#include "sc_common.cuh"

namespace {

template <typename T> struct Vec8;  // 8 consecutive elements
template <> struct Vec8<float> {
  float v[8];
  struct Raw { float4 a, b; };
  static __device__ __forceinline__ Raw load_raw(const float* p) { Raw r; r.a = *(const float4*)p; r.b = *(const float4*)(p + 4); return r; }
  __device__ __forceinline__ void from_raw(const Raw& r) {
    v[0] = r.a.x; v[1] = r.a.y; v[2] = r.a.z; v[3] = r.a.w; v[4] = r.b.x; v[5] = r.b.y; v[6] = r.b.z; v[7] = r.b.w;
  }
  __device__ __forceinline__ void load(const float* p) {
    float4 a = *(const float4*)p, b = *(const float4*)(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  __device__ __forceinline__ void store(float* p) const {
    *(float4*)p = make_float4(v[0], v[1], v[2], v[3]);
    *(float4*)(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
};
template <> struct Vec8<__nv_bfloat16> {
  float v[8];
  struct Raw { uint4 u; };
  static __device__ __forceinline__ Raw load_raw(const __nv_bfloat16* p) { Raw r; r.u = *(const uint4*)p; return r; }
  __device__ __forceinline__ void from_raw(const Raw& r) {
    const uint32_t w[4] = {r.u.x, r.u.y, r.u.z, r.u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ __forceinline__ void load(const __nv_bfloat16* p) {
    uint4 u = *(const uint4*)p;
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ __forceinline__ void store(__nv_bfloat16* p) const {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *(uint32_t*)&t;
    }
    *(uint4*)p = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

__device__ __forceinline__ float group_sum(float x, int lanes) {
  for (int o = lanes >> 1; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// ---------------------------------------------------------------------------------------------------------
// K5: thread = (row, 8-dim chunk); dk/8 adjacent lanes form a head.  Appends k_t,v_t to slot n_prev and attends over
// slots 0..n_prev with an online softmax (keys stream through registers, 16-byte loads, 1 KB coalesced per row).
// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256, 3) self_attn_step_kernel(const T* __restrict__ q, const T* __restrict__ k,
                                                             const T* __restrict__ v, int ldq, int ldk, int ldv,
                                                             T* __restrict__ cache_k, T* __restrict__ cache_v,
                                                             const int* __restrict__ anc, int anc_ld, int slot_div,
                                                             T* __restrict__ out, int ldo, int R, int D, int dk,
                                                             int n_prev, int write_slot) {
  const int chunks = D / 8;
  const int lanes = dk / 8;
  sc::pdl_wait();
  const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = g < (long)R * chunks;
  const int r = active ? (int)(g / chunks) : R - 1;
  const int c = active ? (int)(g % chunks) : 0;
  const float scale_div = sqrtf((float)dk);
  Vec8<T> qv, kv, vv;
  qv.load(q + (size_t)r * ldq + c * 8);
  kv.load(k + (size_t)r * ldk + c * 8);
  vv.load(v + (size_t)r * ldv + c * 8);
  if (active && write_slot >= 0) {
    kv.store(cache_k + ((size_t)write_slot * R + r) * D + c * 8);
    vv.store(cache_v + ((size_t)write_slot * R + r) * D + c * 8);
  }
  float m = -INFINITY, l = 0.f, acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  // one online-softmax update (same operation order as a plain loop over the slots: results are bit-identical)
  auto update = [&](const Vec8<T>& kk, const Vec8<T>& vs) {
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) dot = fmaf(qv.v[i], kk.v[i], dot);
    dot = group_sum(dot, lanes) / scale_div;
    const float mn = fmaxf(m, dot);
    const float corr = expf(m - mn);
    const float p = expf(dot - mn);
    l = l * corr + p;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = acc[i] * corr + p * vs.v[i];
    m = mn;
  };
  // The slot loop was a chain of dependent round trips (ancestor index -> K, V -> update -> next slot: ~0.6 us each, 12.5 us
  // at t = 15 for 50 MB, 62 % of the HBM rate).  Four slots are now requested together before any of them is consumed.
  constexpr int kAhead = 4;
  for (int s0 = 0; s0 < n_prev; s0 += kAhead) {
    int src[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) src[u] = (s0 + u < n_prev) ? anc[(size_t)r * anc_ld + (s0 + u) / slot_div] : 0;
    typename Vec8<T>::Raw kr[kAhead], vr[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      if (s0 + u < n_prev) {
        kr[u] = Vec8<T>::load_raw(cache_k + ((size_t)(s0 + u) * R + src[u]) * D + c * 8);
        vr[u] = Vec8<T>::load_raw(cache_v + ((size_t)(s0 + u) * R + src[u]) * D + c * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      if (s0 + u < n_prev) {  // block-uniform
        Vec8<T> kk, vs;
        kk.from_raw(kr[u]); vs.from_raw(vr[u]);
        update(kk, vs);
      }
    }
  }
  update(kv, vv);  // the current token
  // the cache has been streamed: only now may the next kernel's CTAs take SM slots (a trigger at the top cost this
  // HBM-bound kernel ~20 % in back-to-back measurements)
  sc::pdl_launch();
  const float inv = 1.f / l;
  Vec8<T> o;
#pragma unroll
  for (int i = 0; i < 8; ++i) o.v[i] = acc[i] * inv;
  if (active) o.store(out + (size_t)r * ldo + c * 8);
}

// ---------------------------------------------------------------------------------------------------------
// K6: one warp per (image, head) serves the NB beam rows of that image together, so each memory K/V element is
// loaded once per image instead of once per beam.  Scores: lane = key (16-byte loads of that key's d_k slice, q
// broadcast from shared memory); softmax by warp shuffles; PV: lane = output dims, V rows read coalesced.
// ---------------------------------------------------------------------------------------------------------
constexpr int kMaxKeyPass = 4;  // N <= 128 memory slots

// 16-byte global -> shared copies of one (image, head) K or V slice: rows of dk elements, row stride in smem = rb bytes
template <typename T>
__device__ __forceinline__ void stage_rows(const T* __restrict__ src, int ld, unsigned char* dst, int rb, int N, int dk, int lane) {
  const int vec_per_row = dk * (int)sizeof(T) / 16;
  const int total = N * vec_per_row;
  for (int e0 = 0; e0 < total; e0 += 32 * 4) {
    uint4 tmp[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {  // 4 loads in flight per lane
      const int e = e0 + u * 32 + lane;
      if (e < total) {
        const int j = e / vec_per_row, c = e - j * vec_per_row;
        tmp[u] = *(const uint4*)((const unsigned char*)(src + (size_t)j * ld) + c * 16);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = e0 + u * 32 + lane;
      if (e < total) {
        const int j = e / vec_per_row, c = e - j * vec_per_row;
        *(uint4*)(dst + (size_t)j * rb + c * 16) = tmp[u];
      }
    }
  }
}

template <typename T, int NB>
__global__ void __launch_bounds__(256) cross_attn_step_kernel(const T* __restrict__ q, int ldq, const T* __restrict__ mk,
                                                              const T* __restrict__ mv, int ldm,
                                                              const float* __restrict__ att_mask, T* __restrict__ out,
                                                              int ldo, int B, int N, int h, int dk, int warps) {
  extern __shared__ __align__(16) unsigned char smem_x[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * warps + warp;
  sc::pdl_launch();
  sc::pdl_wait();
  if (w >= B * h) return;
  const int b = w / h, hh = w - b * h;
  const int rbk = dk * (int)sizeof(T) + 16;  // padded K rows: lane=key 16-byte reads are bank-conflict free
  const int rbv = dk * (int)sizeof(T);
  const int per_warp = N * (rbk + rbv) + NB * dk * 4;
  unsigned char* base = smem_x + (size_t)warp * per_warp;
  unsigned char* sk = base;
  unsigned char* sv = base + (size_t)N * rbk;
  float* sq = (float*)(sv + (size_t)N * rbv);
  stage_rows<T>(mk + (size_t)b * N * ldm + hh * dk, ldm, sk, rbk, N, dk, lane);
  stage_rows<T>(mv + (size_t)b * N * ldm + hh * dk, ldm, sv, rbv, N, dk, lane);
  for (int e = lane; e < NB * dk; e += 32) {
    const int n = e / dk, d = e - n * dk;
    sq[e] = sc::to_f32<T>(q[((size_t)b * NB + n) * ldq + hh * dk + d]);
  }
  __syncwarp();
  const float scale_div = sqrtf((float)dk);
  float sc_[kMaxKeyPass][NB];
  float mx[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) mx[n] = -INFINITY;
#pragma unroll
  for (int ps = 0; ps < kMaxKeyPass; ++ps) {
    const int j = ps * 32 + lane;
    float dot[NB];
#pragma unroll
    for (int n = 0; n < NB; ++n) dot[n] = 0.f;
    if (ps * 32 < N && j < N) {
      const T* kr = (const T*)(sk + (size_t)j * rbk);
      for (int c = 0; c < dk; c += 8) {
        Vec8<T> kk;
        kk.load(kr + c);
#pragma unroll
        for (int n = 0; n < NB; ++n) {
          const float4 q0 = *(const float4*)(sq + n * dk + c), q1 = *(const float4*)(sq + n * dk + c + 4);
          dot[n] = fmaf(q0.x, kk.v[0], dot[n]); dot[n] = fmaf(q0.y, kk.v[1], dot[n]);
          dot[n] = fmaf(q0.z, kk.v[2], dot[n]); dot[n] = fmaf(q0.w, kk.v[3], dot[n]);
          dot[n] = fmaf(q1.x, kk.v[4], dot[n]); dot[n] = fmaf(q1.y, kk.v[5], dot[n]);
          dot[n] = fmaf(q1.z, kk.v[6], dot[n]); dot[n] = fmaf(q1.w, kk.v[7], dot[n]);
        }
      }
      const bool masked = att_mask && att_mask[(size_t)b * N + j] == 0.f;
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        float sv_ = dot[n] / scale_div;
        if (masked) sv_ = -1e9f;
        sc_[ps][n] = sv_;
        mx[n] = fmaxf(mx[n], sv_);
      }
    } else {
#pragma unroll
      for (int n = 0; n < NB; ++n) sc_[ps][n] = -INFINITY;
    }
  }
  float inv[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const float m = sc::warp_max(mx[n]);
    float sum = 0.f;
#pragma unroll
    for (int ps = 0; ps < kMaxKeyPass; ++ps) {
      const float e = (ps * 32 + lane < N) ? expf(sc_[ps][n] - m) : 0.f;
      sc_[ps][n] = e;
      sum += e;
    }
    inv[n] = 1.f / sc::warp_sum(sum);
  }
  // PV: lane owns dims lane, lane+32 (d_k <= 64); V rows come from shared memory
  float o0[NB], o1[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) { o0[n] = 0.f; o1[n] = 0.f; }
  const bool d0 = lane < dk, d1 = lane + 32 < dk;
#pragma unroll
  for (int ps = 0; ps < kMaxKeyPass; ++ps) {
    if (ps * 32 >= N) break;
    const int lim = min(32, N - ps * 32);
    for (int l = 0; l < lim; ++l) {
      const T* vr = (const T*)(sv + (size_t)(ps * 32 + l) * rbv);
      const float v0 = d0 ? sc::to_f32<T>(vr[lane]) : 0.f;
      const float v1 = d1 ? sc::to_f32<T>(vr[lane + 32]) : 0.f;
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        const float p = __shfl_sync(0xffffffffu, sc_[ps][n], l);
        o0[n] = fmaf(p, v0, o0[n]);
        o1[n] = fmaf(p, v1, o1[n]);
      }
    }
  }
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    T* orow = out + ((size_t)b * NB + n) * ldo + hh * dk;
    if (d0) orow[lane] = sc::from_f32<T>(o0[n] * inv[n]);
    if (d1) orow[lane + 32] = sc::from_f32<T>(o1[n] * inv[n]);
  }
}

// kWideChunk query rows (q rows row0 .. row0 + kWideChunk - 1, of which the first nq exist) of cross_attn_step_wide_kernel
// against the K/V slice staged at sk / sv: the scores, softmax and PV of cross_attn_step_kernel<T, kWideChunk>, rows n < nq
// written to out.  (A copy rather than a helper shared with that kernel: sharing changed the register allocation of the
// <= 8-beam instantiations.)
constexpr int kWideChunk = 8;
template <typename T>
__device__ __forceinline__ void cross_attn_rows(const T* __restrict__ q, int ldq, const float* __restrict__ att_mask,
                                                T* __restrict__ out, int ldo, size_t row0, int nq, const unsigned char* sk,
                                                const unsigned char* sv, float* sq, int rbk, int rbv, int b, int N, int hh,
                                                int dk, int lane) {
  constexpr int NB = kWideChunk;
  for (int e = lane; e < NB * dk; e += 32) {
    const int n = e / dk, d = e - n * dk;
    sq[e] = n < nq ? sc::to_f32<T>(q[(row0 + n) * ldq + hh * dk + d]) : 0.f;
  }
  __syncwarp();
  const float scale_div = sqrtf((float)dk);
  float sc_[kMaxKeyPass][NB];
  float mx[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) mx[n] = -INFINITY;
#pragma unroll
  for (int ps = 0; ps < kMaxKeyPass; ++ps) {
    const int j = ps * 32 + lane;
    float dot[NB];
#pragma unroll
    for (int n = 0; n < NB; ++n) dot[n] = 0.f;
    if (ps * 32 < N && j < N) {
      const T* kr = (const T*)(sk + (size_t)j * rbk);
      for (int c = 0; c < dk; c += 8) {
        Vec8<T> kk;
        kk.load(kr + c);
#pragma unroll
        for (int n = 0; n < NB; ++n) {
          const float4 q0 = *(const float4*)(sq + n * dk + c), q1 = *(const float4*)(sq + n * dk + c + 4);
          dot[n] = fmaf(q0.x, kk.v[0], dot[n]); dot[n] = fmaf(q0.y, kk.v[1], dot[n]);
          dot[n] = fmaf(q0.z, kk.v[2], dot[n]); dot[n] = fmaf(q0.w, kk.v[3], dot[n]);
          dot[n] = fmaf(q1.x, kk.v[4], dot[n]); dot[n] = fmaf(q1.y, kk.v[5], dot[n]);
          dot[n] = fmaf(q1.z, kk.v[6], dot[n]); dot[n] = fmaf(q1.w, kk.v[7], dot[n]);
        }
      }
      const bool masked = att_mask && att_mask[(size_t)b * N + j] == 0.f;
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        float sv_ = dot[n] / scale_div;
        if (masked) sv_ = -1e9f;
        sc_[ps][n] = sv_;
        mx[n] = fmaxf(mx[n], sv_);
      }
    } else {
#pragma unroll
      for (int n = 0; n < NB; ++n) sc_[ps][n] = -INFINITY;
    }
  }
  float inv[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const float m = sc::warp_max(mx[n]);
    float sum = 0.f;
#pragma unroll
    for (int ps = 0; ps < kMaxKeyPass; ++ps) {
      const float e = (ps * 32 + lane < N) ? expf(sc_[ps][n] - m) : 0.f;
      sc_[ps][n] = e;
      sum += e;
    }
    inv[n] = 1.f / sc::warp_sum(sum);
  }
  // PV: lane owns dims lane, lane+32 (d_k <= 64); V rows come from shared memory
  float o0[NB], o1[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) { o0[n] = 0.f; o1[n] = 0.f; }
  const bool d0 = lane < dk, d1 = lane + 32 < dk;
#pragma unroll
  for (int ps = 0; ps < kMaxKeyPass; ++ps) {
    if (ps * 32 >= N) break;
    const int lim = min(32, N - ps * 32);
    for (int l = 0; l < lim; ++l) {
      const T* vr = (const T*)(sv + (size_t)(ps * 32 + l) * rbv);
      const float v0 = d0 ? sc::to_f32<T>(vr[lane]) : 0.f;
      const float v1 = d1 ? sc::to_f32<T>(vr[lane + 32]) : 0.f;
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        const float p = __shfl_sync(0xffffffffu, sc_[ps][n], l);
        o0[n] = fmaf(p, v0, o0[n]);
        o1[n] = fmaf(p, v1, o1[n]);
      }
    }
  }
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    if (n >= nq) break;
    T* orow = out + (row0 + n) * ldo + hh * dk;
    if (d0) orow[lane] = sc::from_f32<T>(o0[n] * inv[n]);
    if (d1) orow[lane + 32] = sc::from_f32<T>(o1[n] * inv[n]);
  }
}

// 9 .. 32 beams: the same per-warp staging of the (image, head) K/V slice, then kWideChunk query rows at a time, so the
// memory K/V are still read from HBM once per image.
template <typename T>
__global__ void __launch_bounds__(256) cross_attn_step_wide_kernel(const T* __restrict__ q, int ldq, const T* __restrict__ mk,
                                                                   const T* __restrict__ mv, int ldm,
                                                                   const float* __restrict__ att_mask, T* __restrict__ out,
                                                                   int ldo, int B, int beam, int N, int h, int dk, int warps) {
  extern __shared__ __align__(16) unsigned char smem_x[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * warps + warp;
  sc::pdl_launch();
  sc::pdl_wait();
  if (w >= B * h) return;
  const int b = w / h, hh = w - b * h;
  const int rbk = dk * (int)sizeof(T) + 16;
  const int rbv = dk * (int)sizeof(T);
  const int per_warp = N * (rbk + rbv) + kWideChunk * dk * 4;
  unsigned char* base = smem_x + (size_t)warp * per_warp;
  unsigned char* sk = base;
  unsigned char* sv = base + (size_t)N * rbk;
  float* sq = (float*)(sv + (size_t)N * rbv);
  stage_rows<T>(mk + (size_t)b * N * ldm + hh * dk, ldm, sk, rbk, N, dk, lane);
  stage_rows<T>(mv + (size_t)b * N * ldm + hh * dk, ldm, sv, rbv, N, dk, lane);
  for (int c = 0; c < beam; c += kWideChunk) {
    __syncwarp();  // the previous chunk's query rows have been read
    cross_attn_rows<T>(q, ldq, att_mask, out, ldo, (size_t)b * beam + c, min(kWideChunk, beam - c), sk, sv, sq,
                                   rbk, rbv, b, N, hh, dk, lane);
  }
}

// ---------------------------------------------------------------------------------------------------------
// K7 beam step.  One CTA per image.
// ---------------------------------------------------------------------------------------------------------
constexpr int kMaxBeam = 8;       // beams served by the per-thread candidate lists below
constexpr int kMaxWideBeam = 32;  // beams served by the radix-select row pass and merge (beam > kMaxBeam)
constexpr int kBeamThreads = 256;
constexpr int kBeamWarps = kBeamThreads / 32;
constexpr int kBeamRegs = 40;  // logits of one row live in registers when V <= 256*40 = 10240

struct Cand {
  float s;
  int idx;  // flat index beam*V + word; smaller index wins ties (== stable descending sort)
};
__device__ __forceinline__ bool better(const Cand& a, const Cand& b) { return a.s > b.s || (a.s == b.s && a.idx < b.idx); }

template <int NB>
__device__ __forceinline__ void topk_insert(Cand (&top)[NB], Cand c) {
  if (!better(c, top[NB - 1])) return;
  top[NB - 1] = c;
#pragma unroll
  for (int i = NB - 1; i > 0; --i) {
    if (better(top[i], top[i - 1])) { Cand t = top[i]; top[i] = top[i - 1]; top[i - 1] = t; }
  }
}

struct BeamArgs {
  const float* logits;  // [B*beam, V] raw generator output (bias included)
  int B, beam, V, L, t;
  int eos, pad;
  float temperature;
  int constraint;      // decoding_constraint: forbid repeating the previous token
  int penalty_kind;    // 0 none, 1 wu, 2 avg
  float penalty_alpha;
  // beam state, ping-pong (in -> out)
  const int* seq_in; int* seq_out;        // [B*beam, L]
  const float* lp_in; float* lp_out;      // [B*beam, L] log-prob of each chosen token
  float* sum;                             // [B*beam] running joint log-prob (in/out)
  const int* anc_in; int* anc_out;        // [B*beam, L]
  int* tokens_out;                        // [B*beam] token fed at step t+1
  // finished beams: running top-`beam` per image
  int* done_seq; float* done_lp; double* done_p; int* done_count;  // [B,beam,L] [B,beam,L] [B,beam] [B]
  // fused generator (sc_beam_step_partials): logits == nullptr; the raw logit of candidate j of row r is ws_raw[r*beam + j]
  const float* ws_raw;
  // remove_bad_endings (caption_model.py:161-168): per-row token whose log-prob is -inf at this step (-1 = none), and
  // suppress_UNK (:169-170): column whose log-prob is lowered by 1000 (-1 = none).  Both act AFTER the normalisation.
  const int* suppress_tok;
  int penalized_col;
  // diverse beam search (sc_beam_step_diverse, caption_model.py:33-52): the candidates of this group are ranked by
  // log-prob - div_lambda * (number of beams of the groups p < div_group whose token at position t is that column).
  // div_hist holds every group's seq ping-pong buffers [G][2][B*beam][L]; t is this group's local step.
  const int* div_hist;
  int div_group;
  float div_lambda;
};

// Diverse beam search: tokens at position a.t of the current beams of groups p < a.div_group for image b.  The groups are
// staggered (group p runs at local step a.t + div_group - p in the same global step and has already taken it, or stopped
// at L-1), so group p's current history is its ping-pong buffer (min(a.t + div_group - p, L-1) + 1) & 1.
__device__ __forceinline__ int diversity_token(const BeamArgs& a, int NB, int b, int i) {
  const int p = i / NB, j = i - p * NB;
  const int tp = min(a.t + a.div_group - p, a.L - 1);
  return a.div_hist[(((size_t)p * 2 + ((tp + 1) & 1)) * a.B * NB + (size_t)b * NB + j) * a.L + a.t];
}

// Block-wide: s_tok[i] = the i-th earlier-group token, s_cnt[i] = its multiplicity at its first occurrence, 0 at repeats.
// Returns the number of entries (div_group * NB <= kBeamThreads).
__device__ __forceinline__ int diversity_table(const BeamArgs& a, int NB, int b, int* s_tok, float* s_cnt) {
  const int n = a.div_group * NB, tid = threadIdx.x;
  int tok = -1;
  if (tid < n) s_tok[tid] = tok = diversity_token(a, NB, b, tid);
  __syncthreads();
  if (tid < n) {
    int c = 0;
    bool first = true;
    for (int i = 0; i < n; ++i) {
      c += s_tok[i] == tok;
      first = first && !(i < tid && s_tok[i] == tok);
    }
    s_cnt[tid] = first ? (float)c : 0.f;
  }
  __syncthreads();
  return n;
}

__device__ __forceinline__ float diversity_count(int col, int n, const int* s_tok, const float* s_cnt) {
  float c = 0.f;
  for (int i = 0; i < n; ++i) c += (s_tok[i] == col) ? s_cnt[i] : 0.f;
  return c;
}

// Smallest penalised column > `after` owned by this thread in a column-strided scan (col % kBeamThreads == threadIdx.x);
// 0x7fffffff when none is left.
__device__ __forceinline__ int diversity_next(int after, int n, const int* s_tok, const float* s_cnt) {
  int best = 0x7fffffff;
  for (int i = 0; i < n; ++i) {
    const int c = s_tok[i];
    if (s_cnt[i] > 0.f && c > after && c < best && c % kBeamThreads == (int)threadIdx.x) best = c;
  }
  return best;
}

__device__ __forceinline__ float block_max(float v, float* s_red) {
  v = sc::warp_max(v);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = s_red[0];
#pragma unroll
  for (int w = 1; w < kBeamWarps; ++w) r = fmaxf(r, s_red[w]);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_sum(float v, float* s_red) {
  v = sc::warp_sum(v);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
#pragma unroll
  for (int w = 0; w < kBeamWarps; ++w) r += s_red[w];
  __syncthreads();
  return r;
}

// Phase A — one CTA per ROW (image, beam): the row is read from HBM exactly once into registers (kRegs: V <= 256*40;
// otherwise re-read through L2), log-softmax statistics, then the row's top-NB candidates by FINAL score
// (sum + log-prob, ties to the smaller flat index == stable descending sort) -> workspace.
// kDiv (diverse beam search): the final score is sum + (log-prob - lambda * count); log-softmax statistics come from the
// row without the penalty, and within the row the score is monotone in x - T * lambda * count (as for suppress_UNK).
template <int NB, bool kRegs, bool kDiv = false>
__global__ void __launch_bounds__(kBeamThreads, 4) beam_row_kernel(const BeamArgs a, float* __restrict__ ws_stats,
                                                                Cand* __restrict__ ws_cand) {
  const int r = blockIdx.x;            // row = b*NB + k
  const int k = r % NB;
  sc::pdl_wait();
  if (a.t == 0 && k != 0) return;      // first step: every beam holds BOS, only beam 0 is expanded
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int V = a.V;
  __shared__ float s_red[kBeamWarps];
  __shared__ Cand s_top[kBeamWarps][NB];
  __shared__ int s_dtok[kDiv ? kBeamThreads : 1];
  __shared__ float s_dcnt[kDiv ? kBeamThreads : 1];
  const int ndiv = kDiv ? diversity_table(a, NB, r / NB, s_dtok, s_dcnt) : 0;
  // init_logprobs (t == 0) are never temperature-scaled (caption_model.py:135, 218)
  const float T = (a.t == 0) ? 1.0f : a.temperature;
  const float* x = a.logits + (size_t)r * V;
  Cand top[NB];
#pragma unroll
  for (int i = 0; i < NB; ++i) { top[i].s = -INFINITY; top[i].idx = 0x7fffffff; }
  const float base = a.sum[r];
  const int prev = (a.constraint && a.t > 0) ? a.seq_in[(size_t)r * a.L + a.t - 1] : -1;
  const int sup = (a.suppress_tok && a.t > 0) ? a.suppress_tok[r] : -1;
  const int pen = a.penalized_col;
  float mx = -INFINITY, ls, mx2 = 0.f, ls2 = 0.f;
  if (kRegs) {
    // Register path (V <= 10240, V % 4 == 0): the row is read once with 16-byte loads.  The kernel used to be
    // issue-bound (~75 instructions per logit: accurate expf + a full score per element); now per logit: one max, one
    // compare against the thread's NB-th best RAW logit, one ex2.approx.  Within a row the final score
    // s = sum + log_softmax(x) is a monotone function of x, so the thread's top-NB by (x, smaller index) are its
    // top-NB by (s, smaller index) unless >= NB+1 candidates collapse to one fp32 score at the cut; exact scores are
    // then computed for the NB survivors only and every merge below ranks by (s, idx) as before.
    float4 xr[kBeamRegs / 4];
    const float4* x4 = (const float4*)x;
    const int V4 = V >> 2;
#pragma unroll
    for (int i = 0; i < kBeamRegs / 4; ++i) {
      const int c4 = tid + i * kBeamThreads;
      xr[i] = c4 < V4 ? __ldg(x4 + c4) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    Cand rawtop[NB];  // .s = raw logit
#pragma unroll
    for (int i = 0; i < NB; ++i) { rawtop[i].s = -INFINITY; rawtop[i].idx = 0x7fffffff; }
#pragma unroll
    for (int i = 0; i < kBeamRegs / 4; ++i) {
      const int c0 = (tid + i * kBeamThreads) * 4;
      float v[4] = {xr[i].x, xr[i].y, xr[i].z, xr[i].w};
      mx = fmaxf(mx, fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])));
      if (prev >= c0 && prev < c0 + 4) v[prev - c0] = -INFINITY;  // decoding_constraint: never a candidate
      if (sup >= c0 && sup < c0 + 4) v[sup - c0] = -INFINITY;
      if (pen >= c0 && pen < c0 + 4) v[pen - c0] -= 1000.f * T;  // log-prob - 1000 (the final score is (x - mx - ls) / T ...)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (v[e] > rawtop[NB - 1].s) {  // ascending index order: strict '>' keeps the smaller index on ties
          Cand cd; cd.s = v[e]; cd.idx = c0 + e;
          topk_insert<NB>(rawtop, cd);
        }
      }
    }
    mx = block_max(mx, s_red);
    sc::pdl_launch();  // the row is in registers: the merge kernel's CTAs may be scheduled
    float se = 0.f;
#pragma unroll
    for (int i = 0; i < kBeamRegs / 4; ++i)
      se += __expf(xr[i].x - mx) + __expf(xr[i].y - mx) + __expf(xr[i].z - mx) + __expf(xr[i].w - mx);  // exp(-inf) = 0
    se = block_sum(se, s_red);
    ls = logf(se);  // torch.log_softmax: lp = (x - max) - log(sum exp(x - max))
    if (T != 1.0f) {
      // reference re-normalises log_softmax(lp / T) for t > 0 (caption_model.py:218); max(lp) = -ls
      mx2 = (0.f - ls) / T;
      float se2 = 0.f;
#pragma unroll
      for (int i = 0; i < kBeamRegs / 4; ++i) {
        se2 += __expf(((xr[i].x - mx) - ls) / T - mx2) + __expf(((xr[i].y - mx) - ls) / T - mx2) +
               __expf(((xr[i].z - mx) - ls) / T - mx2) + __expf(((xr[i].w - mx) - ls) / T - mx2);
      }
      ls2 = logf(block_sum(se2, s_red));
    }
    if (kDiv) {
      // The scan above ranked unpenalised logits.  A thread that owns a penalised column (at most g*bdash of the 256) ranks
      // its columns again by x - T * lambda * count, re-read through L1 now that the row's registers are free; the other
      // threads' lists hold no penalised column and stand.
      bool owner = false;
      for (int d = 0; d < ndiv; ++d) owner |= s_dcnt[d] > 0.f && (s_dtok[d] >> 2) % kBeamThreads == tid;
      if (owner) {
#pragma unroll
        for (int i = 0; i < NB; ++i) { rawtop[i].s = -INFINITY; rawtop[i].idx = 0x7fffffff; }
        for (int c0 = tid * 4; c0 < V; c0 += kBeamThreads * 4) {
          for (int e = 0; e < 4; ++e) {
            const int col = c0 + e;
            float v = __ldg(x + col);
            if (col == prev || col == sup) v = -INFINITY;
            if (col == pen) v -= 1000.f * T;
            v -= T * a.div_lambda * diversity_count(col, ndiv, s_dtok, s_dcnt);
            if (v > rawtop[NB - 1].s) {  // ascending index order: strict '>' keeps the smaller index on ties
              Cand cd; cd.s = v; cd.idx = col;
              topk_insert<NB>(rawtop, cd);
            }
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      if (rawtop[i].idx != 0x7fffffff && rawtop[i].s > -INFINITY) {
        float lp;
        if (kDiv) {
          // exact score of the survivor from its unpenalised logit: (log-prob [- 1000]) - lambda * count
          const int col = rawtop[i].idx;
          lp = (__ldg(x + col) - mx) - ls;
          if (T != 1.0f) lp = (lp / T - mx2) - ls2;
          if (col == pen) lp -= 1000.f;
          lp = __fsub_rn(lp, __fmul_rn(a.div_lambda, diversity_count(col, ndiv, s_dtok, s_dcnt)));
        } else {
          lp = (rawtop[i].s - mx) - ls;
          if (T != 1.0f) lp = (lp / T - mx2) - ls2;
        }
        Cand cd; cd.s = base + lp; cd.idx = k * V + rawtop[i].idx;
        topk_insert<NB>(top, cd);
      }
    }
  } else {
    for (int i = tid; i < V; i += kBeamThreads) mx = fmaxf(mx, x[i]);
    mx = block_max(mx, s_red);
    float se = 0.f;
    for (int i = tid; i < V; i += kBeamThreads) se += __expf(x[i] - mx);
    se = block_sum(se, s_red);
    ls = logf(se);
    if (T != 1.0f) {
      mx2 = (0.f - ls) / T;
      float se2 = 0.f;
      for (int i = tid; i < V; i += kBeamThreads) se2 += __expf(((x[i] - mx) - ls) / T - mx2);
      ls2 = logf(block_sum(se2, s_red));
    }
    // kDiv: the thread walks its own penalised columns in ascending order next to the scan (O(V) plus O(g*bdash) per hit)
    int next_pen = kDiv ? diversity_next(-1, ndiv, s_dtok, s_dcnt) : -1;
    for (int i = tid; i < V; i += kBeamThreads) {
      float lp = (x[i] - mx) - ls;
      if (T != 1.0f) lp = (lp / T - mx2) - ls2;
      if (i == prev || i == sup) lp = -INFINITY;
      if (i == pen) lp -= 1000.f;
      if (kDiv && i == next_pen) {
        lp = __fsub_rn(lp, __fmul_rn(a.div_lambda, diversity_count(i, ndiv, s_dtok, s_dcnt)));
        next_pen = diversity_next(i, ndiv, s_dtok, s_dcnt);
      }
      Cand cd; cd.s = base + lp; cd.idx = k * V + i;
      topk_insert<NB>(top, cd);
    }
  }
  if (tid == 0) {
    ws_stats[r * 4 + 0] = mx; ws_stats[r * 4 + 1] = ls; ws_stats[r * 4 + 2] = mx2; ws_stats[r * 4 + 3] = ls2;
  }
  // warp merge: every lane offers its sorted list; NB rounds of arg-best over the heads
  {
    int head = 0;
#pragma unroll
    for (int rnd = 0; rnd < NB; ++rnd) {
      Cand c;
      c.s = -INFINITY; c.idx = 0x7fffffff;
#pragma unroll
      for (int i = 0; i < NB; ++i) if (i == head) c = top[i];
      Cand best = c;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        Cand other;
        other.s = __shfl_xor_sync(0xffffffffu, best.s, o);
        other.idx = __shfl_xor_sync(0xffffffffu, best.idx, o);
        if (better(other, best)) best = other;
      }
      if (head < NB && c.idx == best.idx && c.s == best.s) head++;
      if (lane == 0) s_top[warp][rnd] = best;
    }
  }
  __syncthreads();
  if (tid == 0) {
    int heads[kBeamWarps];
#pragma unroll
    for (int w = 0; w < kBeamWarps; ++w) heads[w] = 0;
    for (int rnd = 0; rnd < NB; ++rnd) {
      int bw = 0;
      Cand best; best.s = -INFINITY; best.idx = 0x7fffffff;
#pragma unroll
      for (int w = 0; w < kBeamWarps; ++w) {
        Cand c; c.s = -INFINITY; c.idx = 0x7fffffff;
        if (heads[w] < NB) c = s_top[w][heads[w]];
        if (better(c, best)) { best = c; bw = w; }
      }
#pragma unroll
      for (int w = 0; w < kBeamWarps; ++w) if (w == bw) heads[w]++;
      ws_cand[(size_t)r * NB + rnd] = best;
    }
  }
}

// Phase A for the fused generator (sc_linear_topk): one WARP per row reduces the row's P records
// {max, sum exp(x - max), kPartTopK largest logits, their columns} to the log-softmax statistics and the row's top-NB
// candidates (same outputs as beam_row_kernel, plus the raw logit of each candidate for the merge kernel).
constexpr int kPartTopK = 5;
constexpr int kPartRec = 2 + 2 * kPartTopK;
// kDiv (diverse beam search, group g of bdash = NB beams): the row keeps its top NB + g*NB <= kPartTopK raw candidates (the
// records must hold that many: sc_linear_topk candidates = the whole beam size); at most g*NB distinct columns are
// penalised, so the top NB by penalised score are among them.
template <int NB, bool kDiv = false>
__global__ void __launch_bounds__(256) beam_row_partials_kernel(const BeamArgs a, const float* __restrict__ part, int P,
                                                                float* __restrict__ ws_stats, Cand* __restrict__ ws_cand,
                                                                float* __restrict__ ws_raw) {
  constexpr int NR = kDiv ? kPartTopK : NB;  // raw candidates kept per row
  sc::pdl_launch();
  sc::pdl_wait();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= a.B * NB) return;
  const int k = r % NB;
  if (a.t == 0 && k != 0) return;  // first step: only beam 0 is expanded
  const float* pr = part + (size_t)r * P * kPartRec;
  // lane-local: running (max, sum) and top-NR by (raw logit, smaller column)
  float m = -INFINITY, sum = 0.f;
  Cand top[NR];
#pragma unroll
  for (int i = 0; i < NR; ++i) { top[i].s = -INFINITY; top[i].idx = 0x7fffffff; }
  for (int p = lane; p < P; p += 32) {
    const float* rec = pr + (size_t)p * kPartRec;
    const float pm = rec[0], ps = rec[1];
    if (pm > -INFINITY) {
      if (pm > m) { sum = sum * __expf(m - pm) + ps; m = pm; }
      else sum += ps * __expf(pm - m);
    }
#pragma unroll
    for (int i = 0; i < kPartTopK; ++i) {
      if (i >= NR) break;  // a record's i-th entry can only matter for i < NR
      Cand cd; cd.s = rec[2 + i]; cd.idx = __float_as_int(rec[2 + kPartTopK + i]);
      if (cd.idx != 0x7fffffff) topk_insert<NR>(top, cd);
    }
  }
  // warp: global max, rescaled sum
  const float M = sc::warp_max(m);
  float sc_ = (m > -INFINITY) ? sum * __expf(m - M) : 0.f;
  sc_ = sc::warp_sum(sc_);
  const float ls = logf(sc_);
  const float base = a.sum[r];
  // warp merge of the lanes' sorted lists (NB rounds of arg-best over the heads), ranking by (raw logit, column) - within
  // a row the final score base + (x - M) - ls is monotone in x
  int head = 0;
  Cand raw[NR];  // the row's top-NR (raw logit, column), warp-uniform
#pragma unroll
  for (int rnd = 0; rnd < NR; ++rnd) {
    Cand c; c.s = -INFINITY; c.idx = 0x7fffffff;
#pragma unroll
    for (int i = 0; i < NR; ++i) if (i == head) c = top[i];
    Cand best = c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      Cand other;
      other.s = __shfl_xor_sync(0xffffffffu, best.s, o);
      other.idx = __shfl_xor_sync(0xffffffffu, best.idx, o);
      if (better(other, best)) best = other;
    }
    if (head < NR && c.idx == best.idx && c.s == best.s) head++;
    raw[rnd] = best;
    if (!kDiv && lane == 0) {
      Cand out; out.s = -INFINITY; out.idx = 0x7fffffff;
      if (best.idx != 0x7fffffff) { out.s = base + ((best.s - M) - ls); out.idx = k * a.V + best.idx; }
      ws_cand[(size_t)r * NB + rnd] = out;
      ws_raw[(size_t)r * NB + rnd] = best.s;
    }
  }
  if (kDiv) {
    // lane i < g*NB holds the i-th earlier-group token; exact penalised scores of the NR raw candidates, then the top NB
    const int n = a.div_group * NB;
    const int tok = lane < n ? diversity_token(a, NB, r / NB, lane) : -1;
    Cand sc[NR];
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      float c = 0.f;
      for (int j = 0; j < n; ++j) c += (__shfl_sync(0xffffffffu, tok, j) == raw[i].idx) ? 1.f : 0.f;
      sc[i].s = -INFINITY; sc[i].idx = 0x7fffffff;
      if (raw[i].idx != 0x7fffffff) {
        sc[i].s = base + __fsub_rn((raw[i].s - M) - ls, __fmul_rn(a.div_lambda, c));
        sc[i].idx = k * a.V + raw[i].idx;
      }
    }
    unsigned used = 0;
#pragma unroll
    for (int rnd = 0; rnd < NB; ++rnd) {
      int bj = 0;
      Cand best; best.s = -INFINITY; best.idx = 0x7fffffff;
#pragma unroll
      for (int i = 0; i < NR; ++i)
        if (!(used >> i & 1u) && better(sc[i], best)) { best = sc[i]; bj = i; }
      used |= 1u << bj;
      if (lane == 0) {
        ws_cand[(size_t)r * NB + rnd] = best;
        ws_raw[(size_t)r * NB + rnd] = raw[bj].s;
      }
    }
  }
  if (lane == 0) { ws_stats[r * 4 + 0] = M; ws_stats[r * 4 + 1] = ls; ws_stats[r * 4 + 2] = 0.f; ws_stats[r * 4 + 3] = 0.f; }
}

// Phase B — one small CTA per image: NB-way merge of the rows' sorted candidate lists, then the beam bookkeeping
// (caption_model.py:84-110, 195-210).
constexpr int kMergeThreads = 64;
template <int NB>
__global__ void __launch_bounds__(kMergeThreads) beam_merge_kernel(const BeamArgs a, const float* __restrict__ ws_stats,
                                                                   const Cand* __restrict__ ws_cand) {
  const int b = blockIdx.x;
  const int tid = threadIdx.x;
  const int V = a.V;
  sc::pdl_launch();
  sc::pdl_wait();
  const int rows = (a.t == 0) ? 1 : NB;
  __shared__ Cand s_final[NB];
  __shared__ int s_src[NB];  // winner j came from candidate slot s_src[j] = row k * NB + position
  __shared__ int s_pos, s_last;
  const float T = (a.t == 0) ? 1.0f : a.temperature;
  if (tid == 0) {
    int heads[NB];
#pragma unroll
    for (int k = 0; k < NB; ++k) heads[k] = 0;
    for (int rnd = 0; rnd < NB; ++rnd) {
      int bk = 0;
      Cand best; best.s = -INFINITY; best.idx = 0x7fffffff;
#pragma unroll
      for (int k = 0; k < NB; ++k) {
        Cand c; c.s = -INFINITY; c.idx = 0x7fffffff;
        if (k < rows && heads[k] < NB) c = ws_cand[((size_t)b * NB + k) * NB + heads[k]];
        if (better(c, best)) { best = c; bk = k; }
      }
#pragma unroll
      for (int k = 0; k < NB; ++k) if (k == bk) { s_src[rnd] = k * NB + heads[k]; heads[k]++; }
      s_final[rnd] = best;
    }
  }
  __syncthreads();

  const int L = a.L, t = a.t;
  for (int e = tid; e < NB * L; e += kMergeThreads) {
    const int j = e / L, s = e - j * L;
    const int parent = s_final[j].idx / V;
    const size_t src = ((size_t)b * NB + parent) * L + s, dst = ((size_t)b * NB + j) * L + s;
    if (s < t) {
      a.seq_out[dst] = a.seq_in[src];
      a.lp_out[dst] = a.lp_in[src];
      a.anc_out[dst] = a.anc_in[src];
    } else if (s == t) {
      const int word = s_final[j].idx - parent * V;
      a.seq_out[dst] = word;
      const float x = a.logits ? a.logits[((size_t)b * NB + parent) * V + word] : a.ws_raw[(size_t)b * NB * NB + s_src[j]];
      const float* st = ws_stats + ((size_t)b * NB + parent) * 4;
      float lp = (x - st[0]) - st[1];
      if (T != 1.0f) lp = (lp / T - st[2]) - st[3];
      if (word == a.penalized_col) lp -= 1000.f;
      a.lp_out[dst] = lp;
      a.anc_out[dst] = b * NB + parent;
    } else {
      a.seq_out[dst] = a.pad;
      a.lp_out[dst] = 0.f;
      a.anc_out[dst] = b * NB + j;  // slots of future steps are written by the row itself
    }
  }
  __syncthreads();
  // finished beams: stable insertion into the running top-NB (python's sorted() is stable and entries arrive
  // chronologically); thread 0 picks the slot, L threads move the rows.
  int cnt = a.done_count[b];
  for (int j = 0; j < NB; ++j) {
    const int parent = s_final[j].idx / V;
    const int word = s_final[j].idx - parent * V;
    float ys = s_final[j].s;
    const bool is_end = (word == a.eos) || (t == L - 1);
    if (is_end) {
      if (tid == 0) {
        // the reference scores finished beams in Python floats (double): model_utils.py:121-146
        double p = (double)ys;
        const double len = (double)(t + 1);
        if (a.penalty_kind == 1) p = p / (pow(5.0 + len, (double)a.penalty_alpha) / pow(6.0, (double)a.penalty_alpha));
        else if (a.penalty_kind == 2) p = p / len;
        int pos = cnt < NB ? cnt : NB;
        while (pos > 0 && a.done_p[b * NB + pos - 1] < p) --pos;
        const int last = (cnt < NB ? cnt : NB - 1);
        if (pos < NB) {
          for (int m = last; m > pos; --m) a.done_p[b * NB + m] = a.done_p[b * NB + m - 1];
          a.done_p[b * NB + pos] = p;
        }
        s_pos = pos; s_last = last;
      }
      __syncthreads();
      const int pos = s_pos, last = s_last;
      if (pos < NB) {
        for (int s = tid; s < L; s += kMergeThreads) {
          for (int m = last; m > pos; --m) {
            a.done_seq[((size_t)b * NB + m) * L + s] = a.done_seq[((size_t)b * NB + m - 1) * L + s];
            a.done_lp[((size_t)b * NB + m) * L + s] = a.done_lp[((size_t)b * NB + m - 1) * L + s];
          }
          const size_t src = ((size_t)b * NB + j) * L + s;
          a.done_seq[((size_t)b * NB + pos) * L + s] = s <= t ? a.seq_out[src] : a.pad;
          a.done_lp[((size_t)b * NB + pos) * L + s] = s <= t ? a.lp_out[src] : 0.f;
        }
        if (cnt < NB) cnt++;
      }
      __syncthreads();
      ys -= 1000.f;
    }
    if (tid == 0) {
      a.tokens_out[b * NB + j] = word;
      a.sum[b * NB + j] = ys;
    }
  }
  if (tid == 0) a.done_count[b] = cnt;
}


// ---------------------------------------------------------------------------------------------------------
// Wide beams (kMaxBeam < beam <= kMaxWideBeam).  A per-thread insertion list of `beam` candidates does not fit in
// registers, so both phases select with a block-wide radix select on 64-bit keys (order-preserving uint32 of the final
// score << 32 | ~flat index): the keys are all distinct and a larger key is a better candidate under `better`, so "every
// key whose digits >= the k-th largest key's" is the exact top-k even with ties and -inf scores.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long cand_key(float s, int idx) {
  uint32_t u = __float_as_uint(s);
  if ((u << 1) == 0u) u = 0u;  // -0.0 keyed as +0.0: equal scores tie on the index
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned long long)(~(uint32_t)idx);
}

struct RadixSmem {
  unsigned hist[256];
  unsigned wsum[kBeamWarps];
  int bin, rem, cnt;
};

// Block-wide (kBeamThreads threads) selection of the k largest of a set of distinct keys; each(f) calls f(key) for every
// key of the calling thread.  A key is among the k largest iff (key & mask) >= prefix.  8-bit digits from the top; the
// passes stop once every key left under the prefix is needed.
struct RadixCut { unsigned long long prefix, mask; };
template <typename Each>
__device__ __forceinline__ RadixCut radix_top(Each each, int k, RadixSmem& sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long prefix = 0ull, mask = 0ull;
  int rem = k;
  for (int shift = 56; shift >= 0; shift -= 8) {
    sm.hist[tid] = 0u;
    __syncthreads();
    each([&](unsigned long long key) {
      if ((key & mask) == prefix) atomicAdd(&sm.hist[(unsigned)(key >> shift) & 255u], 1u);
    });
    __syncthreads();
    // inclusive scan from the top digit down: incl = keys under the prefix whose digit >= 255 - tid
    const unsigned c = sm.hist[255 - tid];
    unsigned incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    if (lane == 31) sm.wsum[warp] = incl;
    __syncthreads();
    for (int w = 0; w < warp; ++w) incl += sm.wsum[w];
    const unsigned excl = incl - c;
    if (excl < (unsigned)rem && incl >= (unsigned)rem) { sm.bin = 255 - tid; sm.rem = rem - (int)excl; sm.cnt = (int)c; }
    __syncthreads();
    prefix |= (unsigned long long)sm.bin << shift;
    mask |= 0xffull << shift;
    rem = sm.rem;
    if (sm.cnt == rem) break;  // block-uniform
  }
  RadixCut cut;
  cut.prefix = prefix; cut.mask = mask;
  return cut;
}

// Phase A for wide beams — one CTA per row, as beam_row_kernel: the row is read once (registers when V <= 256*40,
// otherwise re-read through L2 on every pass), the log-softmax statistics, then the exact final score of every column.
// The `beam`-th largest of the threads' best keys bounds the row's `beam`-th largest key from below, so only the keys above
// it (a few times `beam` in practice) enter the radix passes.  The row's top-`beam` candidates go to the workspace unsorted.
template <bool kRegs>
__global__ void __launch_bounds__(kBeamThreads, 4) beam_row_wide_kernel(const BeamArgs a, float* __restrict__ ws_stats,
                                                                       Cand* __restrict__ ws_cand) {
  const int beam = a.beam;
  const int r = blockIdx.x;  // row = b*beam + k
  const int k = r % beam;
  sc::pdl_wait();
  if (a.t == 0 && k != 0) return;  // first step: every beam holds BOS, only beam 0 is expanded
  const int tid = threadIdx.x;
  const int V = a.V;
  __shared__ float s_red[kBeamWarps];
  __shared__ RadixSmem s_rs;
  __shared__ unsigned long long s_best[kBeamThreads];
  __shared__ unsigned long long s_floor;
  __shared__ int s_n;
  const float T = (a.t == 0) ? 1.0f : a.temperature;
  const float* x = a.logits + (size_t)r * V;
  const float base = a.sum[r];
  const int prev = (a.constraint && a.t > 0) ? a.seq_in[(size_t)r * a.L + a.t - 1] : -1;
  const int sup = (a.suppress_tok && a.t > 0) ? a.suppress_tok[r] : -1;
  const int pen = a.penalized_col;
  const int flat0 = k * V;
  float mx = -INFINITY, ls, mx2 = 0.f, ls2 = 0.f;
  // final score of column col (the order of operations of beam_row_kernel's L2 path)
  auto score = [&](float v, int col) {
    float lp = (v - mx) - ls;
    if (T != 1.0f) lp = (lp / T - mx2) - ls2;
    if (col == prev || col == sup) lp = -INFINITY;
    if (col == pen) lp -= 1000.f;
    return base + lp;
  };
  float4 xr[kRegs ? kBeamRegs / 4 : 1];
  if constexpr (kRegs) {
    const float4* x4 = (const float4*)x;
    const int V4 = V >> 2;
#pragma unroll
    for (int i = 0; i < kBeamRegs / 4; ++i) {
      const int c4 = tid + i * kBeamThreads;
      xr[i] = c4 < V4 ? __ldg(x4 + c4) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      mx = fmaxf(mx, fmaxf(fmaxf(xr[i].x, xr[i].y), fmaxf(xr[i].z, xr[i].w)));
    }
    mx = block_max(mx, s_red);
    sc::pdl_launch();  // the row is in registers: the merge kernel's CTAs may be scheduled
    float se = 0.f;
#pragma unroll
    for (int i = 0; i < kBeamRegs / 4; ++i)
      se += __expf(xr[i].x - mx) + __expf(xr[i].y - mx) + __expf(xr[i].z - mx) + __expf(xr[i].w - mx);
    ls = logf(block_sum(se, s_red));
    if (T != 1.0f) {
      mx2 = (0.f - ls) / T;
      float se2 = 0.f;
#pragma unroll
      for (int i = 0; i < kBeamRegs / 4; ++i) {
        se2 += __expf(((xr[i].x - mx) - ls) / T - mx2) + __expf(((xr[i].y - mx) - ls) / T - mx2) +
               __expf(((xr[i].z - mx) - ls) / T - mx2) + __expf(((xr[i].w - mx) - ls) / T - mx2);
      }
      ls2 = logf(block_sum(se2, s_red));
    }
#pragma unroll
    for (int i = 0; i < kBeamRegs / 4; ++i) {  // the registers now hold final scores
      const int c0 = (tid + i * kBeamThreads) * 4;
      xr[i].x = score(xr[i].x, c0); xr[i].y = score(xr[i].y, c0 + 1);
      xr[i].z = score(xr[i].z, c0 + 2); xr[i].w = score(xr[i].w, c0 + 3);
    }
  } else {
    for (int i = tid; i < V; i += kBeamThreads) mx = fmaxf(mx, x[i]);
    mx = block_max(mx, s_red);
    float se = 0.f;
    for (int i = tid; i < V; i += kBeamThreads) se += __expf(x[i] - mx);
    ls = logf(block_sum(se, s_red));
    if (T != 1.0f) {
      mx2 = (0.f - ls) / T;
      float se2 = 0.f;
      for (int i = tid; i < V; i += kBeamThreads) se2 += __expf(((x[i] - mx) - ls) / T - mx2);
      ls2 = logf(block_sum(se2, s_red));
    }
  }
  // f(key, score, column) for every column of this thread
  auto each_col = [&](auto f) {
    if constexpr (kRegs) {
#pragma unroll
      for (int i = 0; i < kBeamRegs / 4; ++i) {
        const int c0 = (tid + i * kBeamThreads) * 4;
        if (c0 < V) {  // V % 4 == 0 on this path
          f(cand_key(xr[i].x, flat0 + c0), xr[i].x, c0); f(cand_key(xr[i].y, flat0 + c0 + 1), xr[i].y, c0 + 1);
          f(cand_key(xr[i].z, flat0 + c0 + 2), xr[i].z, c0 + 2); f(cand_key(xr[i].w, flat0 + c0 + 3), xr[i].w, c0 + 3);
        }
      }
    } else {
      for (int i = tid; i < V; i += kBeamThreads) {
        const float s = score(__ldg(x + i), i);
        f(cand_key(s, flat0 + i), s, i);
      }
    }
  };
  // floor = the beam-th largest of the threads' best keys (0 = no key: then every key passes)
  unsigned long long best = 0ull;
  each_col([&](unsigned long long key, float, int) { best = key > best ? key : best; });
  s_best[tid] = best;
  if (tid == 0) { s_floor = 0ull; s_n = 0; }
  __syncthreads();
  int above = 0;
  for (int j = 0; j < kBeamThreads; ++j) above += s_best[j] > best;
  if (above == beam - 1) s_floor = best;
  __syncthreads();
  const unsigned long long floor_key = s_floor;
  const RadixCut cut = radix_top(
      [&](auto f) {
        each_col([&](unsigned long long key, float, int) {
          if (key >= floor_key) f(key);
        });
      },
      beam, s_rs);
  each_col([&](unsigned long long key, float s, int col) {
    if (key >= floor_key && (key & cut.mask) >= cut.prefix) {
      Cand cd; cd.s = s; cd.idx = flat0 + col;
      ws_cand[(size_t)r * beam + atomicAdd(&s_n, 1)] = cd;
    }
  });
  if (tid == 0) {
    ws_stats[r * 4 + 0] = mx; ws_stats[r * 4 + 1] = ls; ws_stats[r * 4 + 2] = mx2; ws_stats[r * 4 + 3] = ls2;
  }
}

// Phase B for wide beams — one CTA per image: the top `beam` of the rows' beam x beam candidates by the same radix select,
// ranked among themselves, then the beam bookkeeping of beam_merge_kernel (a copy rather than a shared helper: sharing
// changed the register allocation of the <= 8-beam merge).
__global__ void __launch_bounds__(kBeamThreads) beam_merge_wide_kernel(const BeamArgs a, const float* __restrict__ ws_stats,
                                                                       const Cand* __restrict__ ws_cand) {
  const int b = blockIdx.x;
  const int tid = threadIdx.x;
  const int beam = a.beam;
  sc::pdl_launch();
  sc::pdl_wait();
  const int n = ((a.t == 0) ? 1 : beam) * beam;
  __shared__ unsigned long long s_key[kMaxWideBeam * kMaxWideBeam];
  __shared__ RadixSmem s_rs;
  __shared__ unsigned long long s_sel[kMaxWideBeam];
  __shared__ int s_sel_src[kMaxWideBeam];
  __shared__ Cand s_final[kMaxWideBeam];
  __shared__ int s_src[kMaxWideBeam];
  __shared__ int s_n, s_pos, s_last;
  const Cand* cand = ws_cand + (size_t)b * beam * beam;
  for (int i = tid; i < n; i += kBeamThreads) s_key[i] = cand_key(cand[i].s, cand[i].idx);
  if (tid == 0) s_n = 0;
  __syncthreads();
  const RadixCut cut = radix_top(
      [&](auto f) {
        for (int i = tid; i < n; i += kBeamThreads) f(s_key[i]);
      },
      beam, s_rs);
  for (int i = tid; i < n; i += kBeamThreads) {
    if ((s_key[i] & cut.mask) >= cut.prefix) {
      const int j = atomicAdd(&s_n, 1);
      s_sel[j] = s_key[i];
      s_sel_src[j] = i;
    }
  }
  __syncthreads();
  if (tid < beam) {
    int rank = 0;
    for (int j = 0; j < beam; ++j) rank += s_sel[j] > s_sel[tid];
    s_final[rank] = cand[s_sel_src[tid]];
    s_src[rank] = s_sel_src[tid];
  }
  __syncthreads();
  // the bookkeeping of beam_merge_kernel with nb = beam winners and kBeamThreads threads
  const int nb = beam;
  const int V = a.V;
  const float T = (a.t == 0) ? 1.0f : a.temperature;
  const int L = a.L, t = a.t;
  for (int e = tid; e < nb * L; e += kBeamThreads) {
    const int j = e / L, s = e - j * L;
    const int parent = s_final[j].idx / V;
    const size_t src = ((size_t)b * nb + parent) * L + s, dst = ((size_t)b * nb + j) * L + s;
    if (s < t) {
      a.seq_out[dst] = a.seq_in[src];
      a.lp_out[dst] = a.lp_in[src];
      a.anc_out[dst] = a.anc_in[src];
    } else if (s == t) {
      const int word = s_final[j].idx - parent * V;
      a.seq_out[dst] = word;
      const float x = a.logits ? a.logits[((size_t)b * nb + parent) * V + word] : a.ws_raw[(size_t)b * nb * nb + s_src[j]];
      const float* st = ws_stats + ((size_t)b * nb + parent) * 4;
      float lp = (x - st[0]) - st[1];
      if (T != 1.0f) lp = (lp / T - st[2]) - st[3];
      if (word == a.penalized_col) lp -= 1000.f;
      a.lp_out[dst] = lp;
      a.anc_out[dst] = b * nb + parent;
    } else {
      a.seq_out[dst] = a.pad;
      a.lp_out[dst] = 0.f;
      a.anc_out[dst] = b * nb + j;  // slots of future steps are written by the row itself
    }
  }
  __syncthreads();
  // finished beams: stable insertion into the running top-nb (python's sorted() is stable and entries arrive
  // chronologically); thread 0 picks the slot, L threads move the rows.
  int cnt = a.done_count[b];
  for (int j = 0; j < nb; ++j) {
    const int parent = s_final[j].idx / V;
    const int word = s_final[j].idx - parent * V;
    float ys = s_final[j].s;
    const bool is_end = (word == a.eos) || (t == L - 1);
    if (is_end) {
      if (tid == 0) {
        // the reference scores finished beams in Python floats (double): model_utils.py:121-146
        double p = (double)ys;
        const double len = (double)(t + 1);
        if (a.penalty_kind == 1) p = p / (pow(5.0 + len, (double)a.penalty_alpha) / pow(6.0, (double)a.penalty_alpha));
        else if (a.penalty_kind == 2) p = p / len;
        int pos = cnt < nb ? cnt : nb;
        while (pos > 0 && a.done_p[b * nb + pos - 1] < p) --pos;
        const int last = (cnt < nb ? cnt : nb - 1);
        if (pos < nb) {
          for (int m = last; m > pos; --m) a.done_p[b * nb + m] = a.done_p[b * nb + m - 1];
          a.done_p[b * nb + pos] = p;
        }
        s_pos = pos; s_last = last;
      }
      __syncthreads();
      const int pos = s_pos, last = s_last;
      if (pos < nb) {
        for (int s = tid; s < L; s += kBeamThreads) {
          for (int m = last; m > pos; --m) {
            a.done_seq[((size_t)b * nb + m) * L + s] = a.done_seq[((size_t)b * nb + m - 1) * L + s];
            a.done_lp[((size_t)b * nb + m) * L + s] = a.done_lp[((size_t)b * nb + m - 1) * L + s];
          }
          const size_t src = ((size_t)b * nb + j) * L + s;
          a.done_seq[((size_t)b * nb + pos) * L + s] = s <= t ? a.seq_out[src] : a.pad;
          a.done_lp[((size_t)b * nb + pos) * L + s] = s <= t ? a.lp_out[src] : 0.f;
        }
        if (cnt < nb) cnt++;
      }
      __syncthreads();
      ys -= 1000.f;
    }
    if (tid == 0) {
      a.tokens_out[b * nb + j] = word;
      a.sum[b * nb + j] = ys;
    }
  }
  if (tid == 0) a.done_count[b] = cnt;
}

// greedy step (beam_size == 1): one warp per row
__global__ void __launch_bounds__(256) greedy_step_kernel(const float* __restrict__ logits, int R, int V, int L, int t,
                                                          int eos, int constraint, int* __restrict__ seq,
                                                          float* __restrict__ seq_lp, int* __restrict__ tokens,
                                                          int* __restrict__ unfinished, int* __restrict__ live_count) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= R) return;
  // reference loop breaks once every row has finished (transformer.py:550-552): later columns stay pad/0
  if (t > 0 && live_count[t - 1] == 0) return;
  const float* x = logits + (size_t)r * V;
  const int prev = (constraint && t > 0) ? seq[(size_t)r * L + t - 1] : -1;  // transformer.py:523-526 uses seq[:, t-1]
  float mx = -INFINITY; int arg = 0x7fffffff;
  for (int i = lane; i < V; i += 32) {
    const float v = (i == prev) ? -INFINITY : x[i];
    if (v > mx) { mx = v; arg = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
  }
  // log-softmax over the unconstrained row
  float rmx = -INFINITY;
  for (int i = lane; i < V; i += 32) rmx = fmaxf(rmx, x[i]);
  rmx = sc::warp_max(rmx);
  float se = 0.f;
  for (int i = lane; i < V; i += 32) se += expf(x[i] - rmx);
  se = sc::warp_sum(se);
  if (lane == 0) {
    const int unf = unfinished[r];
    seq[(size_t)r * L + t] = unf ? arg : 0;
    seq_lp[(size_t)r * L + t] = mx - (rmx + logf(se));
    const int still = unf && (arg != eos);
    unfinished[r] = still;
    tokens[r] = arg;
    if (still) atomicAdd(&live_count[t], 1);
  }
}

// multinomial step (num_random_sample > 0, models/transformer.py:531-538): it ~ Categorical(exp(logprobs / T)), the stored
// log-prob is the un-tempered log_softmax entry.  One warp per row; inverse CDF in index order: the sampled token is the
// first i with sum_{j<=i} w_j > u * sum_j w_j, u = uniforms[r] (tests) or Philox(seed, stream t, row).
__global__ void __launch_bounds__(256) sample_step_kernel(const float* __restrict__ logits, int R, int V, int L, int t, int eos,
                                                          int constraint, float inv_T, const float* __restrict__ uniforms,
                                                          unsigned long long seed, int* __restrict__ seq,
                                                          float* __restrict__ seq_lp, int* __restrict__ tokens,
                                                          int* __restrict__ unfinished, int* __restrict__ live_count) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= R) return;
  if (t > 0 && live_count[t - 1] == 0) return;
  const float* x = logits + (size_t)r * V;
  const int prev = (constraint && t > 0) ? seq[(size_t)r * L + t - 1] : -1;
  float rmx = -INFINITY;
  for (int i = lane; i < V; i += 32) rmx = fmaxf(rmx, x[i]);
  rmx = sc::warp_max(rmx);
  float se = 0.f;
  for (int i = lane; i < V; i += 32) se += expf(x[i] - rmx);
  se = sc::warp_sum(se);
  const float lse = rmx + logf(se);
  float tot = 0.f;
  // weights relative to the row maximum: exp((lp_i - lp_max) / T) - the same distribution as exp(lp_i / T), without the
  // underflow of small temperatures
  for (int i = lane; i < V; i += 32) tot += (i == prev) ? 0.f : expf((x[i] - rmx) * inv_T);
  tot = sc::warp_sum(tot);
  float u;
  if (uniforms) u = uniforms[r];
  else { const sc::Philox ph(seed); u = sc::u24(ph((uint64_t)r, (uint64_t)t).x); }
  const float thr = u * tot;
  float cum = 0.f;
  int pick = -1;
  for (int base = 0; base < V && pick < 0; base += 32) {
    const int i = base + lane;
    float w = (i < V && i != prev) ? expf((x[i] - rmx) * inv_T) : 0.f;
    float sc_ = w;  // inclusive scan over the 32 lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float n = __shfl_up_sync(0xffffffffu, sc_, o);
      if (lane >= o) sc_ += n;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, w > 0.f && cum + sc_ > thr);
    if (hit) pick = base + __ffs(hit) - 1;
    cum += __shfl_sync(0xffffffffu, sc_, 31);
  }
  // rounding can leave the threshold a hair above the accumulated total: take the last admissible token
  if (pick < 0) pick = (V - 1 == prev) ? V - 2 : V - 1;
  if (lane == 0) {
    const int unf = unfinished[r];
    seq[(size_t)r * L + t] = unf ? pick : 0;
    seq_lp[(size_t)r * L + t] = x[pick] - lse;
    const int still = unf && (pick != eos);
    unfinished[r] = still;
    tokens[r] = pick;
    if (still) atomicAdd(&live_count[t], 1);
  }
}

// K8: dst[r] = src[idx[r]] for rows of row_bytes (16-byte vectorised)
__global__ void __launch_bounds__(256) reorder_rows_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst,
                                                           const int* __restrict__ idx, long rows, long vec_per_row) {
  const long total = rows * vec_per_row;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long)gridDim.x * blockDim.x) {
    const long r = g / vec_per_row, c = g - r * vec_per_row;
    dst[g] = src[(long)idx[r] * vec_per_row + c];
  }
}

}  // namespace

// tensor-path cross-attention (sc_mma_attention.cu); SC_ERR_UNSUPPORTED = shape not served, nothing launched
int sc_cross_attn_mma_launch(const void* q, int ldq, const void* mem_k, const void* mem_v, int ldm, const float* att_mask,
                             void* out, int ldo, int B, int beam, int N, int h, cudaStream_t stream);

extern "C" {

int sc_decode_self_attn_step(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int dtype,
                             void* cache_k, void* cache_v, const int* anc, int anc_ld, int slot_div, void* out, int ldo,
                             int R, int D, int h, int n_prev, int write_slot, cudaStream_t stream) {
  SC_CHECK(R > 0 && D > 0 && h > 0 && D % h == 0, SC_ERR_SHAPE, "sc_decode_self_attn_step: R=%d D=%d h=%d", R, D, h);
  const int dk = D / h;
  SC_CHECK(dk % 8 == 0 && dk <= 256 && (dk & (dk - 1)) == 0, SC_ERR_UNSUPPORTED,
           "sc_decode_self_attn_step: d_k=%d must be a power of two in [8,256]", dk);
  SC_CHECK(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0, SC_ERR_ALIGN, "sc_decode_self_attn_step: ld %% 8");
  SC_CHECK(n_prev >= 0 && slot_div >= 1, SC_ERR_SHAPE, "sc_decode_self_attn_step: n_prev=%d slot_div=%d", n_prev, slot_div);
  SC_CHECK(n_prev == 0 || anc != nullptr, SC_ERR_SHAPE, "sc_decode_self_attn_step: ancestor table missing");
  const long threads = (long)R * (D / 8);
  const int blocks = (int)((threads + 255) / 256);
  if (dtype == SC_F32)
    sc::launch_pdl(self_attn_step_kernel<float>, dim3(blocks), dim3(256), 0, stream, (const float*)q, (const float*)k,
                   (const float*)v, ldq, ldk, ldv, (float*)cache_k, (float*)cache_v, anc, anc_ld, slot_div, (float*)out, ldo, R, D,
                   dk, n_prev, write_slot);
  else if (dtype == SC_BF16)
    sc::launch_pdl(self_attn_step_kernel<__nv_bfloat16>, dim3(blocks), dim3(256), 0, stream, (const __nv_bfloat16*)q,
                   (const __nv_bfloat16*)k, (const __nv_bfloat16*)v, ldq, ldk, ldv, (__nv_bfloat16*)cache_k,
                   (__nv_bfloat16*)cache_v, anc, anc_ld, slot_div, (__nv_bfloat16*)out, ldo, R, D, dk, n_prev, write_slot);
  else
    SC_CHECK(false, SC_ERR_DTYPE, "sc_decode_self_attn_step: bad dtype %d", dtype);
  SC_LAUNCH_CHECK("sc_decode_self_attn_step");
  return SC_OK;
}

int sc_decode_cross_attn_step(const void* q, int ldq, const void* mem_k, const void* mem_v, int ldm, int dtype,
                              const float* att_mask, void* out, int ldo, int B, int beam, int N, int D, int h,
                              cudaStream_t stream) {
  SC_CHECK(B > 0 && beam > 0 && N > 0 && D % h == 0, SC_ERR_SHAPE, "sc_decode_cross_attn_step: bad shape");
  const int dk = D / h;
  SC_CHECK(dk % 8 == 0 && dk <= 256 && (dk & (dk - 1)) == 0, SC_ERR_UNSUPPORTED,
           "sc_decode_cross_attn_step: d_k=%d must be a power of two in [8,256]", dk);
  SC_CHECK(ldq % 8 == 0 && ldm % 8 == 0 && ldo % 8 == 0, SC_ERR_ALIGN, "sc_decode_cross_attn_step: ld %% 8");
  SC_CHECK(beam <= kMaxWideBeam, SC_ERR_UNSUPPORTED, "sc_decode_cross_attn_step: beam=%d > %d", beam, kMaxWideBeam);
  SC_CHECK(N <= 32 * kMaxKeyPass, SC_ERR_UNSUPPORTED, "sc_decode_cross_attn_step: N=%d > %d memory slots", N, 32 * kMaxKeyPass);
  SC_CHECK(dk <= 64, SC_ERR_UNSUPPORTED, "sc_decode_cross_attn_step: d_k=%d > 64", dk);
  if (dtype == SC_BF16 && dk == 64) {
    const int rc = sc_cross_attn_mma_launch(q, ldq, mem_k, mem_v, ldm, att_mask, out, ldo, B, beam, N, h, stream);
    if (rc != SC_ERR_UNSUPPORTED) return rc;
  }
  const int esz = dtype == SC_F32 ? 4 : 2;
  const size_t per_warp = (size_t)N * (2 * dk * esz + 16) + (size_t)(beam > kMaxBeam ? kWideChunk : beam) * dk * 4;
  int warps = (int)((96 * 1024) / per_warp);
  if (warps > 8) warps = 8;
  SC_CHECK(warps >= 1, SC_ERR_UNSUPPORTED, "sc_decode_cross_attn_step: N=%d too large for shared memory", N);
  const int blocks = (B * h + warps - 1) / warps;
  const size_t smem = per_warp * warps;
  SC_CHECK(ldm * esz % 16 == 0 && dk * esz % 16 == 0, SC_ERR_ALIGN, "sc_decode_cross_attn_step: 16-byte rows needed");
#define XATT(T, NBV)                                                                                                    \
  do {                                                                                                                  \
    static bool attr_##NBV = false;                                                                                     \
    if (!attr_##NBV) {                                                                                                  \
      cudaFuncSetAttribute(cross_attn_step_kernel<T, NBV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);    \
      attr_##NBV = true;                                                                                                \
    }                                                                                                                   \
    sc::launch_pdl(cross_attn_step_kernel<T, NBV>, dim3(blocks), dim3(32 * warps), smem, stream, (const T*)q, ldq,      \
                   (const T*)mem_k, (const T*)mem_v, ldm, att_mask, (T*)out, ldo, B, N, h, dk, warps);                  \
  } while (0)
#define XATT_NB(T)                                          \
  switch (beam) {                                           \
    case 1: XATT(T, 1); break; case 2: XATT(T, 2); break;   \
    case 3: XATT(T, 3); break; case 4: XATT(T, 4); break;   \
    case 5: XATT(T, 5); break; case 6: XATT(T, 6); break;   \
    case 7: XATT(T, 7); break; default: XATT(T, 8); break;  \
  }
#define XATT_WIDE(T)                                                                                                   \
  do {                                                                                                                 \
    static bool attr_w = false;                                                                                        \
    if (!attr_w) {                                                                                                     \
      cudaFuncSetAttribute(cross_attn_step_wide_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);   \
      attr_w = true;                                                                                                   \
    }                                                                                                                  \
    sc::launch_pdl(cross_attn_step_wide_kernel<T>, dim3(blocks), dim3(32 * warps), smem, stream, (const T*)q, ldq,     \
                   (const T*)mem_k, (const T*)mem_v, ldm, att_mask, (T*)out, ldo, B, beam, N, h, dk, warps);           \
  } while (0)
  if (beam > kMaxBeam && dtype == SC_F32) XATT_WIDE(float);
  else if (beam > kMaxBeam && dtype == SC_BF16) XATT_WIDE(__nv_bfloat16);
  else if (dtype == SC_F32) { XATT_NB(float) }
  else if (dtype == SC_BF16) { XATT_NB(__nv_bfloat16) }
  else SC_CHECK(false, SC_ERR_DTYPE, "sc_decode_cross_attn_step: bad dtype %d", dtype);
#undef XATT_WIDE
#undef XATT_NB
#undef XATT
  SC_LAUNCH_CHECK("sc_decode_cross_attn_step");
  return SC_OK;
}

size_t sc_beam_step_workspace_bytes_impl(int B, int beam) {
  // row statistics [R][4] | candidates [R][beam] | raw logits of the candidates [R][beam] (fused generator path)
  return (size_t)B * beam * (4 * sizeof(float) + (size_t)beam * sizeof(Cand) + (size_t)beam * sizeof(float));
}

// Row pass + merge over materialised logits; a.div_hist != nullptr selects the diverse-beam row pass.
static int beam_step_launch(const char* name, const BeamArgs& a, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  const int B = a.B, beam = a.beam, V = a.V, L = a.L, t = a.t;
  const bool div = a.div_hist != nullptr;
  const int max_beam = div ? kMaxBeam : kMaxWideBeam;  // diverse beam search: beams per group
  SC_CHECK(B > 0 && beam >= 1 && beam <= max_beam, SC_ERR_UNSUPPORTED, "%s: beam=%d not in [1,%d]", name, beam, max_beam);
  SC_CHECK(V >= beam && L > 0 && t >= 0 && t < L, SC_ERR_SHAPE, "%s: V=%d L=%d t=%d", name, V, L, t);
  SC_CHECK(a.temperature > 0.f, SC_ERR_SHAPE, "%s: temperature must be > 0", name);
  SC_CHECK(workspace != nullptr && ((uintptr_t)workspace & 15) == 0 && workspace_bytes >= sc_beam_step_workspace_bytes_impl(B, beam),
           SC_ERR_WORKSPACE, "%s: workspace of %zu bytes (16-byte aligned) needed, got %zu", name,
           sc_beam_step_workspace_bytes_impl(B, beam), workspace_bytes);
  float* ws_stats = (float*)workspace;
  Cand* ws_cand = (Cand*)(ws_stats + (size_t)B * beam * 4);
  const bool regs = V <= kBeamThreads * kBeamRegs && (V & 3) == 0 && ((uintptr_t)a.logits & 15) == 0;
  if (beam > kMaxBeam) {
    if (regs) sc::launch_pdl(beam_row_wide_kernel<true>, dim3(B * beam), dim3(kBeamThreads), 0, stream, a, ws_stats, ws_cand);
    else sc::launch_pdl(beam_row_wide_kernel<false>, dim3(B * beam), dim3(kBeamThreads), 0, stream, a, ws_stats, ws_cand);
    sc::launch_pdl(beam_merge_wide_kernel, dim3(B), dim3(kBeamThreads), 0, stream, a, (const float*)ws_stats, (const Cand*)ws_cand);
    SC_LAUNCH_CHECK(name);
    return SC_OK;
  }
#define BEAM_LAUNCH(NBV)                                                                                                     \
  do {                                                                                                                        \
    if (div && regs) sc::launch_pdl(beam_row_kernel<NBV, true, true>, dim3(B * NBV), dim3(kBeamThreads), 0, stream, a, ws_stats, ws_cand);   \
    else if (div) sc::launch_pdl(beam_row_kernel<NBV, false, true>, dim3(B * NBV), dim3(kBeamThreads), 0, stream, a, ws_stats, ws_cand);    \
    else if (regs) sc::launch_pdl(beam_row_kernel<NBV, true>, dim3(B * NBV), dim3(kBeamThreads), 0, stream, a, ws_stats, ws_cand);          \
    else sc::launch_pdl(beam_row_kernel<NBV, false>, dim3(B * NBV), dim3(kBeamThreads), 0, stream, a, ws_stats, ws_cand);                   \
    sc::launch_pdl(beam_merge_kernel<NBV>, dim3(B), dim3(kMergeThreads), 0, stream, a, ws_stats, (const Cand*)ws_cand);                   \
  } while (0)
  switch (beam) {
    case 1: BEAM_LAUNCH(1); break;
    case 2: BEAM_LAUNCH(2); break;
    case 3: BEAM_LAUNCH(3); break;
    case 4: BEAM_LAUNCH(4); break;
    case 5: BEAM_LAUNCH(5); break;
    case 6: BEAM_LAUNCH(6); break;
    case 7: BEAM_LAUNCH(7); break;
    default: BEAM_LAUNCH(8); break;
  }
#undef BEAM_LAUNCH
  SC_LAUNCH_CHECK(name);
  return SC_OK;
}

static BeamArgs beam_args(const float* logits, int B, int beam, int V, int L, int t, int eos, int pad, float temperature,
                          int decoding_constraint, int penalty_kind, float penalty_alpha, const int* suppress_tok, int penalized_col,
                          const int* seq_in, int* seq_out, const float* lp_in, float* lp_out, float* sum, const int* anc_in,
                          int* anc_out, int* tokens_out, int* done_seq, float* done_lp, double* done_p, int* done_count) {
  BeamArgs a;
  a.logits = logits; a.B = B; a.beam = beam; a.V = V; a.L = L; a.t = t; a.eos = eos; a.pad = pad;
  a.temperature = temperature; a.constraint = decoding_constraint; a.penalty_kind = penalty_kind;
  a.penalty_alpha = penalty_alpha; a.seq_in = seq_in; a.seq_out = seq_out; a.lp_in = lp_in; a.lp_out = lp_out;
  a.sum = sum; a.anc_in = anc_in; a.anc_out = anc_out; a.tokens_out = tokens_out; a.done_seq = done_seq;
  a.done_lp = done_lp; a.done_p = done_p; a.done_count = done_count; a.ws_raw = nullptr;
  a.suppress_tok = suppress_tok; a.penalized_col = (penalized_col >= 0 && penalized_col < V) ? penalized_col : -1;
  a.div_hist = nullptr; a.div_group = 0; a.div_lambda = 0.f;
  return a;
}

int sc_beam_step(const float* logits, int B, int beam, int V, int L, int t, int eos, int pad, float temperature,
                 int decoding_constraint, int penalty_kind, float penalty_alpha, const int* suppress_tok, int penalized_col,
                 const int* seq_in, int* seq_out,
                 const float* lp_in, float* lp_out, float* sum, const int* anc_in, int* anc_out, int* tokens_out,
                 int* done_seq, float* done_lp, double* done_p, int* done_count, void* workspace, size_t workspace_bytes,
                 cudaStream_t stream) {
  const BeamArgs a = beam_args(logits, B, beam, V, L, t, eos, pad, temperature, decoding_constraint, penalty_kind, penalty_alpha,
                               suppress_tok, penalized_col, seq_in, seq_out, lp_in, lp_out, sum, anc_in, anc_out, tokens_out,
                               done_seq, done_lp, done_p, done_count);
  return beam_step_launch("sc_beam_step", a, workspace, workspace_bytes, stream);
}

int sc_beam_step_diverse(const float* logits, int B, int beam, int V, int L, int t, int eos, int pad, float temperature,
                         int decoding_constraint, int penalty_kind, float penalty_alpha, const int* suppress_tok, int penalized_col,
                         const int* group_seq, int group, float diversity_lambda, const int* seq_in, int* seq_out,
                         const float* lp_in, float* lp_out, float* sum, const int* anc_in, int* anc_out, int* tokens_out,
                         int* done_seq, float* done_lp, double* done_p, int* done_count, void* workspace, size_t workspace_bytes,
                         cudaStream_t stream) {
  SC_CHECK(group_seq != nullptr && group >= 0 && group * beam <= kBeamThreads, SC_ERR_SHAPE,
           "sc_beam_step_diverse: group=%d x beam=%d earlier-group beams (at most %d)", group, beam, kBeamThreads);
  BeamArgs a = beam_args(logits, B, beam, V, L, t, eos, pad, temperature, decoding_constraint, penalty_kind, penalty_alpha,
                         suppress_tok, penalized_col, seq_in, seq_out, lp_in, lp_out, sum, anc_in, anc_out, tokens_out,
                         done_seq, done_lp, done_p, done_count);
  a.div_hist = group_seq; a.div_group = group; a.div_lambda = diversity_lambda;
  return beam_step_launch("sc_beam_step_diverse", a, workspace, workspace_bytes, stream);
}

// Beam step from the records of sc_linear_topk instead of materialised logits (temperature 1, no decoding constraint,
// beam <= 5 = the record's candidate count; other options: run sc_linear + sc_beam_step).
static int beam_step_partials_launch(const char* name, BeamArgs& a, const float* partials, int parts_per_row, void* workspace,
                                     size_t workspace_bytes, cudaStream_t stream) {
  const int B = a.B, beam = a.beam, V = a.V, L = a.L, t = a.t;
  SC_CHECK(B > 0 && beam >= 1 && beam <= kPartTopK, SC_ERR_UNSUPPORTED, "%s: beam=%d not in [1,%d]", name, beam, kPartTopK);
  SC_CHECK(V >= beam && L > 0 && t >= 0 && t < L && parts_per_row > 0 && partials != nullptr, SC_ERR_SHAPE,
           "%s: V=%d L=%d t=%d parts=%d", name, V, L, t, parts_per_row);
  SC_CHECK(workspace != nullptr && ((uintptr_t)workspace & 15) == 0 && workspace_bytes >= sc_beam_step_workspace_bytes_impl(B, beam),
           SC_ERR_WORKSPACE, "%s: workspace of %zu bytes (16-byte aligned) needed, got %zu", name,
           sc_beam_step_workspace_bytes_impl(B, beam), workspace_bytes);
  float* ws_stats = (float*)workspace;
  Cand* ws_cand = (Cand*)(ws_stats + (size_t)B * beam * 4);
  float* ws_raw = (float*)(ws_cand + (size_t)B * beam * beam);
  a.ws_raw = ws_raw;
  const int R = B * beam;
  const bool div = a.div_hist != nullptr;
#define BEAMP_LAUNCH(NBV)                                                                                                   \
  do {                                                                                                                       \
    if (div) sc::launch_pdl(beam_row_partials_kernel<NBV, true>, dim3((R + 7) / 8), dim3(256), 0, stream, a, partials, parts_per_row, ws_stats, ws_cand, ws_raw); \
    else sc::launch_pdl(beam_row_partials_kernel<NBV>, dim3((R + 7) / 8), dim3(256), 0, stream, a, partials, parts_per_row, ws_stats, ws_cand, ws_raw); \
    sc::launch_pdl(beam_merge_kernel<NBV>, dim3(B), dim3(kMergeThreads), 0, stream, a, (const float*)ws_stats, (const Cand*)ws_cand); \
  } while (0)
  switch (beam) {
    case 1: BEAMP_LAUNCH(1); break;
    case 2: BEAMP_LAUNCH(2); break;
    case 3: BEAMP_LAUNCH(3); break;
    case 4: BEAMP_LAUNCH(4); break;
    default: BEAMP_LAUNCH(5); break;
  }
#undef BEAMP_LAUNCH
  SC_LAUNCH_CHECK(name);
  return SC_OK;
}

int sc_beam_step_partials(const float* partials, int parts_per_row, int B, int beam, int V, int L, int t, int eos, int pad,
                          int penalty_kind, float penalty_alpha, const int* seq_in, int* seq_out, const float* lp_in,
                          float* lp_out, float* sum, const int* anc_in, int* anc_out, int* tokens_out, int* done_seq,
                          float* done_lp, double* done_p, int* done_count, void* workspace, size_t workspace_bytes,
                          cudaStream_t stream) {
  BeamArgs a = beam_args(nullptr, B, beam, V, L, t, eos, pad, 1.0f, 0, penalty_kind, penalty_alpha, nullptr, -1, seq_in, seq_out,
                         lp_in, lp_out, sum, anc_in, anc_out, tokens_out, done_seq, done_lp, done_p, done_count);
  return beam_step_partials_launch("sc_beam_step_partials", a, partials, parts_per_row, workspace, workspace_bytes, stream);
}

int sc_beam_step_partials_diverse(const float* partials, int parts_per_row, int B, int beam, int V, int L, int t, int eos, int pad,
                                  int penalty_kind, float penalty_alpha, const int* group_seq, int group, float diversity_lambda,
                                  const int* seq_in, int* seq_out, const float* lp_in, float* lp_out, float* sum,
                                  const int* anc_in, int* anc_out, int* tokens_out, int* done_seq, float* done_lp, double* done_p,
                                  int* done_count, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  SC_CHECK(group_seq != nullptr && group >= 0 && (group + 1) * beam <= kPartTopK, SC_ERR_UNSUPPORTED,
           "sc_beam_step_partials_diverse: (group=%d + 1) x beam=%d raw candidates per row exceed the record's %d", group, beam,
           kPartTopK);
  BeamArgs a = beam_args(nullptr, B, beam, V, L, t, eos, pad, 1.0f, 0, penalty_kind, penalty_alpha, nullptr, -1, seq_in, seq_out,
                         lp_in, lp_out, sum, anc_in, anc_out, tokens_out, done_seq, done_lp, done_p, done_count);
  a.div_hist = group_seq; a.div_group = group; a.div_lambda = diversity_lambda;
  return beam_step_partials_launch("sc_beam_step_partials_diverse", a, partials, parts_per_row, workspace, workspace_bytes, stream);
}

int sc_beam_step_workspace_bytes(int B, int beam) { return (int)sc_beam_step_workspace_bytes_impl(B, beam); }

int sc_greedy_step(const float* logits, int R, int V, int L, int t, int eos, int decoding_constraint, int* seq,
                   float* seq_lp, int* tokens, int* unfinished, int* live_count, cudaStream_t stream) {
  SC_CHECK(R > 0 && V > 0 && t >= 0 && t < L, SC_ERR_SHAPE, "sc_greedy_step: R=%d V=%d t=%d L=%d", R, V, t, L);
  greedy_step_kernel<<<(R * 32 + 255) / 256, 256, 0, stream>>>(logits, R, V, L, t, eos, decoding_constraint, seq, seq_lp,
                                                              tokens, unfinished, live_count);
  SC_LAUNCH_CHECK("sc_greedy_step");
  return SC_OK;
}

int sc_sample_step(const float* logits, int R, int V, int L, int t, int eos, int decoding_constraint, float temperature,
                   const float* uniforms, unsigned long long seed, int* seq, float* seq_lp, int* tokens, int* unfinished,
                   int* live_count, cudaStream_t stream) {
  SC_CHECK(R > 0 && V > 1 && t >= 0 && t < L && temperature > 0.f, SC_ERR_SHAPE, "sc_sample_step: R=%d V=%d t=%d L=%d T=%f", R, V, t, L,
           temperature);
  sample_step_kernel<<<(R * 32 + 255) / 256, 256, 0, stream>>>(logits, R, V, L, t, eos, decoding_constraint, 1.0f / temperature,
                                                              uniforms, seed, seq, seq_lp, tokens, unfinished, live_count);
  SC_LAUNCH_CHECK("sc_sample_step");
  return SC_OK;
}

int sc_cache_reorder(const void* src, void* dst, const int* idx, long rows, long row_bytes, cudaStream_t stream) {
  SC_CHECK(rows > 0 && row_bytes > 0 && row_bytes % 16 == 0, SC_ERR_ALIGN, "sc_cache_reorder: row_bytes=%ld must be a multiple of 16", row_bytes);
  SC_CHECK(((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0 && src != dst, SC_ERR_ALIGN, "sc_cache_reorder: alignment / in-place");
  const long vec = row_bytes / 16;
  long blocks = (rows * vec + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  reorder_rows_kernel<<<(int)blocks, 256, 0, stream>>>((const uint4*)src, (uint4*)dst, idx, rows, vec);
  SC_LAUNCH_CHECK("sc_cache_reorder");
  return SC_OK;
}

}  // extern "C"
