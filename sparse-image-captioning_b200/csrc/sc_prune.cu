// Magnitude / SNIP mask updates (sparse_caption/pruning/prune.py:259-289 update_masks_once + compute_mask) on flat buffers.
//
//   sc_prune_stats  : per-segment (sum x, sum x^2) in double, deterministic (per-CTA partials, then a fixed-order reduction);
//                     with `center` (the sums of a first call) the second column is sum (x - mean)^2 instead: the _DIST variance in
//                     two passes, exactly 0 for a constant tensor (so its criterion is 0/0 = NaN whatever the value).
//                     Feeds the _DIST mean / population std, the SNIP normaliser and the per-tensor mask sparsities.
//   sc_prune_select : exact radix select of the k-th smallest (criterion, position) pair per selection group, then the complete
//                     0/1 mask of every segment.  The criterion is computed on the fly from the source buffer in every pass
//                     (no materialised copy): one read of 4 bytes per element per pass, the same traffic a scratch buffer
//                     would cost, and no extra 4 bytes per element of memory.
//
// Keys: the fp32 criterion mapped to an order-preserving uint32 (-0.0 keyed as +0.0, every NaN as one key above +inf, torch's
// sort order), concatenated with the element's 32-bit position in its group: 64-bit keys that are all distinct, so "prune the
// first k in (criterion, position) order" is "prune every key <= the k-th smallest key".  Eight passes of 8-bit digits; a
// group stops as soon as its remaining rank falls on the last element of a digit bucket (continuous criteria: after the four
// criterion bytes), later passes of that group return at once.  Every launch is fixed on the host: no readback, capturable.
#include "sc_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kPerThread = 32;
constexpr int kChunk = kThreads * kPerThread;   // elements per CTA (one segment per CTA)

#define SC_PRUNE_ABS 0
#define SC_PRUNE_DIST 1
#define SC_PRUNE_SNIP 2

struct Seg { long long src_off, dst_off, n, group, pos_base, first_block; };
struct GroupState { unsigned long long prefix; long long k_rem; long long done; long long pad; };

__device__ __forceinline__ int find_seg(const Seg* __restrict__ d, int n_desc, long long b) {
  int lo = 0, hi = n_desc - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (d[mid].first_block <= b) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__device__ __forceinline__ uint32_t order_key(float c) {
  if (c != c) return 0xFFC00000u;                 // NaN: above +inf (0xFF800000)
  uint32_t u = __float_as_uint(c);
  if ((u << 1) == 0u) u = 0u;                     // -0.0 -> +0.0
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// p: DIST {mean, std} of the segment, SNIP {sum of the group's saliency, -}
__device__ __forceinline__ float criterion(int mode, float x, float2 p) {
  if (mode == SC_PRUNE_ABS) return fabsf(x);
  if (mode == SC_PRUNE_DIST) return fabsf(__fdiv_rn(__fsub_rn(x, p.x), p.y));
  return __fdiv_rn(x, p.x);
}

__device__ __forceinline__ unsigned long long full_key(int mode, float x, float2 p, long long pos) {
  return ((unsigned long long)order_key(criterion(mode, x, p)) << 32) | (unsigned long long)(uint32_t)pos;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(kThreads) stats_partial_kernel(const Seg* __restrict__ d, int n_desc, const float* __restrict__ src,
                                                                 int binarize, const double* __restrict__ center,
                                                                 double* __restrict__ partials) {
  const int si = find_seg(d, n_desc, blockIdx.x);
  const Seg s = d[si];
  const double mean = center ? center[2 * si] / (double)s.n : 0.0;
  const long long start = ((long long)blockIdx.x - s.first_block) * kChunk;
  const long long end = min(s.n, start + kChunk);
  double a = 0.0, b = 0.0;
  for (long long i = start + threadIdx.x; i < end; i += kThreads) {
    float x = __ldg(src + s.src_off + i);
    if (binarize) x = sc::mask_round(x);
    a += (double)x;
    const double c = (double)x - mean;
    b += c * c;
  }
  __shared__ double red[2][kThreads / 32];
  a = warp_sum_d(a);
  b = warp_sum_d(b);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    a = b = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) { a += red[0][w]; b += red[1][w]; }
    partials[2 * blockIdx.x] = a;
    partials[2 * blockIdx.x + 1] = b;
  }
}

// one thread per segment, its CTAs' partials in block order
__global__ void stats_reduce_kernel(const Seg* __restrict__ d, int n_desc, long long total_blocks, const double* __restrict__ partials,
                                    double* __restrict__ sums) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_desc; i += gridDim.x * blockDim.x) {
    const long long b1 = i + 1 < n_desc ? d[i + 1].first_block : total_blocks;
    double a = 0.0, b = 0.0;
    for (long long blk = d[i].first_block; blk < b1; ++blk) { a += partials[2 * blk]; b += partials[2 * blk + 1]; }
    sums[2 * i] = a;
    sums[2 * i + 1] = b;
  }
}

// group states from k, zeroed histograms, per-segment criterion parameters
__global__ void select_init_kernel(const Seg* __restrict__ d, int n_desc, int n_groups, const long long* __restrict__ group_k, int mode,
                                   const double* __restrict__ sums, float2* __restrict__ params, GroupState* __restrict__ st,
                                   unsigned* __restrict__ hist) {
  for (int g = threadIdx.x; g < n_groups; g += blockDim.x) {
    const long long k = group_k[g];
    st[g] = GroupState{0ull, k - 1, k <= 0 ? 1ll : 0ll, 0ll};   // k == 0: nothing pruned
  }
  for (int j = threadIdx.x; j < n_groups * 256; j += blockDim.x) hist[j] = 0u;
  for (int i = threadIdx.x; i < n_desc; i += blockDim.x) {
    float2 p = make_float2(0.f, 1.f);
    if (mode == SC_PRUNE_DIST) {
      const double n = (double)d[i].n;   // (sums of the centred pass: second column = sum (x - mean)^2)
      p = make_float2((float)(sums[2 * i] / n), (float)sqrt(sums[2 * i + 1] / n));
    } else if (mode == SC_PRUNE_SNIP) {
      double t = 0.0;   // the whole group's sum, in segment order (every CTA of the group sees the same value)
      for (int j = 0; j < n_desc; ++j)
        if (d[j].group == d[i].group) t += sums[2 * j];
      p.x = (float)t;
    }
    params[i] = p;
  }
}

// digit histogram of the keys that still match their group's prefix (bits above `shift`)
__global__ void __launch_bounds__(kThreads) select_hist_kernel(const Seg* __restrict__ d, int n_desc, int mode, const float* __restrict__ src,
                                                               const float2* __restrict__ params, const GroupState* __restrict__ st,
                                                               unsigned* __restrict__ hist, int shift) {
  const int si = find_seg(d, n_desc, blockIdx.x);
  const Seg s = d[si];
  const GroupState g = st[s.group];
  if (g.done) return;
  __shared__ unsigned h[256];
  h[threadIdx.x] = 0u;
  const float2 p = params[si];
  const long long start = ((long long)blockIdx.x - s.first_block) * kChunk;
  float v[kPerThread];
#pragma unroll
  for (int it = 0; it < kPerThread; ++it) {
    const long long i = start + it * kThreads + threadIdx.x;
    v[it] = i < s.n ? __ldg(src + s.src_off + i) : 0.f;
  }
  __syncthreads();
  const bool top = shift >= 56;
  const unsigned long long want = top ? 0ull : (g.prefix >> (shift + 8));
#pragma unroll
  for (int it = 0; it < kPerThread; ++it) {
    const long long i = start + it * kThreads + threadIdx.x;
    int bin = -1;
    if (i < s.n) {
      const unsigned long long key = full_key(mode, v[it], p, s.pos_base + i);
      if (top || (key >> (shift + 8)) == want) bin = (int)((key >> shift) & 255u);
    }
    // warp-aggregated: the criterion's top byte is the same for most of a tensor
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[bin], (unsigned)__popc(peers));
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&hist[s.group * 256 + threadIdx.x], h[threadIdx.x]);
}

// one CTA per group: the bucket holding the remaining rank, then the histogram is cleared for the next pass
__global__ void __launch_bounds__(256) select_pick_kernel(GroupState* __restrict__ st, unsigned* __restrict__ hist, int shift) {
  GroupState* g = st + blockIdx.x;
  unsigned* h = hist + blockIdx.x * 256;
  const GroupState cur = *g;
  if (cur.done) return;
  const unsigned long long c = h[threadIdx.x];
  h[threadIdx.x] = 0u;
  unsigned long long incl = c;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  __shared__ unsigned long long tot[8];
  if (lane == 31) tot[warp] = incl;
  __syncthreads();
  for (int w = 0; w < warp; ++w) incl += tot[w];
  const unsigned long long excl = incl - c;
  const unsigned long long k = (unsigned long long)cur.k_rem;
  if (c > 0 && excl <= k && k < incl) {
    const unsigned long long kn = k - excl;
    unsigned long long prefix = cur.prefix | ((unsigned long long)threadIdx.x << shift);
    const bool done = kn == c - 1;   // the rank is the bucket's last key: every key of the bucket is pruned
    if (done && shift > 0) prefix |= (1ull << shift) - 1ull;
    *g = GroupState{prefix, (long long)kn, done ? 1ll : 0ll, 0ll};
  }
}

__global__ void __launch_bounds__(kThreads) select_write_kernel(const Seg* __restrict__ d, int n_desc, int mode, const float* __restrict__ src,
                                                                const float2* __restrict__ params, const GroupState* __restrict__ st,
                                                                float* __restrict__ out) {
  const int si = find_seg(d, n_desc, blockIdx.x);
  const Seg s = d[si];
  const GroupState g = st[s.group];
  const bool none = g.k_rem < 0;
  const float2 p = params[si];
  const long long start = ((long long)blockIdx.x - s.first_block) * kChunk;
  const long long end = min(s.n, start + kChunk);
  for (long long i = start + threadIdx.x; i < end; i += kThreads) {
    const bool pruned = !none && full_key(mode, __ldg(src + s.src_off + i), p, s.pos_base + i) <= g.prefix;
    out[s.dst_off + i] = pruned ? 0.f : 1.f;
  }
}

}  // namespace

extern "C" {

int sc_prune_chunk(void) { return kChunk; }

int sc_prune_stats(const void* descs, int n_desc, long total_blocks, const float* src, int binarize, const double* center,
                   double* partials, double* sums, cudaStream_t stream) {
  SC_CHECK(n_desc > 0 && total_blocks > 0, SC_ERR_SHAPE, "sc_prune_stats: n_desc=%d total_blocks=%ld", n_desc, total_blocks);
  SC_CHECK(descs && src && partials && sums, SC_ERR_SHAPE, "sc_prune_stats: null argument");
  const Seg* d = (const Seg*)descs;
  stats_partial_kernel<<<(unsigned)total_blocks, kThreads, 0, stream>>>(d, n_desc, src, binarize, center, partials);
  SC_LAUNCH_CHECK("sc_prune_stats");
  stats_reduce_kernel<<<(n_desc + 127) / 128, 128, 0, stream>>>(d, n_desc, total_blocks, partials, sums);
  SC_LAUNCH_CHECK("sc_prune_stats");
  return SC_OK;
}

int sc_prune_select(const void* descs, int n_desc, long total_blocks, int n_groups, const long long* group_k, int criterion,
                    const float* src, const double* sums, float* mask_out, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  SC_CHECK(n_desc > 0 && total_blocks > 0 && n_groups > 0, SC_ERR_SHAPE, "sc_prune_select: n_desc=%d total_blocks=%ld n_groups=%d",
           n_desc, total_blocks, n_groups);
  SC_CHECK(criterion >= SC_PRUNE_ABS && criterion <= SC_PRUNE_SNIP, SC_ERR_UNSUPPORTED, "sc_prune_select: criterion %d", criterion);
  SC_CHECK(descs && group_k && src && mask_out && workspace, SC_ERR_SHAPE, "sc_prune_select: null argument");
  SC_CHECK(criterion == SC_PRUNE_ABS || sums, SC_ERR_SHAPE, "sc_prune_select: criterion %d needs the segment sums", criterion);
  const size_t need = (size_t)n_groups * (sizeof(GroupState) + 256 * sizeof(unsigned)) + (size_t)n_desc * sizeof(float2);
  SC_CHECK(workspace_bytes >= need && ((uintptr_t)workspace & 15) == 0, SC_ERR_WORKSPACE,
           "sc_prune_select: workspace %zu bytes (16-byte aligned) < %zu", workspace_bytes, need);
  GroupState* st = (GroupState*)workspace;
  unsigned* hist = (unsigned*)(st + n_groups);
  float2* params = (float2*)(hist + (size_t)n_groups * 256);
  const Seg* d = (const Seg*)descs;
  select_init_kernel<<<1, 256, 0, stream>>>(d, n_desc, n_groups, group_k, criterion, sums, params, st, hist);
  SC_LAUNCH_CHECK("sc_prune_select");
  for (int shift = 56; shift >= 0; shift -= 8) {
    select_hist_kernel<<<(unsigned)total_blocks, kThreads, 0, stream>>>(d, n_desc, criterion, src, params, st, hist, shift);
    SC_LAUNCH_CHECK("sc_prune_select");
    select_pick_kernel<<<n_groups, 256, 0, stream>>>(st, hist, shift);
    SC_LAUNCH_CHECK("sc_prune_select");
  }
  select_write_kernel<<<(unsigned)total_blocks, kThreads, 0, stream>>>(d, n_desc, criterion, src, params, st, mask_out);
  SC_LAUNCH_CHECK("sc_prune_select");
  return SC_OK;
}

}  // extern "C"
