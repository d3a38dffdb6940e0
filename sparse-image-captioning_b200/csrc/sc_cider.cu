// Caption scores on the device, on word ids: the CIDEr-D reward of self-critical sequence training (SURVEY.md section 8f.4) and
// the coco-caption validation metrics BLEU-1..4, ROUGE-L and CIDEr.
// CIDEr-D reference: sparse_caption/scst/cider/pyciderevalcap/ciderD/ciderD_scorer.py:133-212 (compute_cider: counts2vec + sim)
// as called by CaptionScorer (sparse_caption/scst/scorers.py:47-114) on decoded sample / baseline captions.  Validation
// metrics reference: pycocoevalcap bleu/bleu_scorer.py (cook_test, compute_score), rouge/rouge.py and cider/cider_scorer.py as
// called by coco_caption/eval.py:15-86 from eval_on_split (utils/training.py:257-327).
//
// The reference detokenises every caption to a string on the host, splits it into words and scores it in Python dictionaries.
// Here the captions stay on the device as word ids: an n-gram (n <= 4) of ids below 65536 is packed exactly into one 64-bit
// key; the document-frequency table (coco-train-words.p in the reference, or the split's own references) and the tf-idf
// vectors / BLEU max counts / token arrays of the reference captions - static over a split - are uploaded once.
// One CTA scores one hypothesis against the references of its image.  All arithmetic is double precision in the reference's
// own summation order (reductions are sequential in first-occurrence n-gram order, like the dict iteration of the reference),
// so scores agree with the Python scorers to the last bits.
#include "sc_common.cuh"

namespace {

constexpr int kMaxWords = 64;
constexpr int kMaxNgrams = 4 * kMaxWords;
constexpr int kThreads = 128;

struct CiderArgs {
  const int* hyp; int L, H;
  const int* hyp_img;
  int eos, pad;
  const unsigned long long* df_keys; const double* df_log; long n_df;   // sorted; df_log = log(max(1, df))
  double ref_len, sigma;
  const long* img_ref_off;      // [B + 1] -> reference captions of an image
  const long* ref_ng_off;       // [R + 1] -> n-gram entries of a reference
  const unsigned long long* ref_keys; const double* ref_vec;   // per reference: keys ascending, tf-idf weights
  const double* ref_norm;       // [R, 4]
  const int* ref_length;        // [R]   (the reference scorer's `length`: its bigram count)
  double* out;                  // [H] (CIDEr-D) or [n_img] indexed by hyp_img (CIDEr)
};

__device__ __forceinline__ long lower_bound(const unsigned long long* a, long n, unsigned long long key) {
  long lo = 0, hi = n;
  while (lo < hi) {
    const long mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

struct BleuArgs {
  const long* img_key_off;                 // [n_img + 1] -> the image's entries of keys / max_count
  const unsigned long long* keys;          // per image: n-gram keys ascending
  const int* max_count;                    // the n-gram's largest count in any one reference of the image
  const long* img_ref_off;                 // [n_img + 1] -> references of an image
  const long* ref_tok_off;                 // [R + 1] -> tokens of a reference (its length is all BLEU needs)
  long long* stats;                        // [n_img, 10]: correct_1..4, guess_1..4, testlen, reflen
  int* hyp_count;                          // [n_img] hypotheses scored per image
  int* bad_index;                          // hypotheses whose image index is outside [0, n_img)
};

enum Metric { kCiderD, kCider, kBleu };

// One CTA per hypothesis.  All three metrics share the n-gram entries of the hypothesis: its words (ids before the first <eos>,
// pads dropped: what tokenizer.decode + str.split leave), one 64-bit key per entry in the reference's dict insertion order
// (k = 1..4, position ascending) and each n-gram's count at its first occurrence.  They are one template rather than a shared
// helper function because an out-of-line helper changes the register allocation of the CIDEr-D instantiation.
//   kCiderD: CIDEr-D (ciderD_scorer.py: clipped hypothesis tf-idf, Gaussian length penalty), out[h].
//   kCider:  coco-caption CIDEr (cider_scorer.py: plain cosine, no penalty), out[hyp_img[h]].
//   kBleu:   the sufficient statistics of bleu_scorer.py cook_test (n = 4, "closest" reference length), b.stats[hyp_img[h]].
// kCider / kBleu skip hypotheses whose image is outside [0, n_img); kBleu counts them and the hypotheses of every image.
template <Metric M>
__global__ void __launch_bounds__(kThreads) ngram_score_kernel(const CiderArgs a, const BleuArgs b, int n_img) {
  __shared__ int s_words[kMaxWords];
  __shared__ unsigned long long s_key[kMaxNgrams];
  __shared__ int s_tf[kMaxNgrams];      // 0 = not the first occurrence of its n-gram (kBleu: the clipped count)
  __shared__ int s_ord[kMaxNgrams];     // n-gram order - 1
  __shared__ double s_vec[kMaxNgrams], s_ref[kMaxNgrams];
  __shared__ double s_norm[4], s_score[4];
  __shared__ int s_nw, s_T;
  const int hI = blockIdx.x, tid = threadIdx.x;
  if constexpr (M != kCiderD) {
    const int img = a.hyp_img[hI];
    if (img < 0 || img >= n_img) {
      if (M == kBleu && tid == 0) atomicAdd(b.bad_index, 1);
      return;
    }
  }
  if (tid == 0) {
    int n = 0;
    for (int i = 0; i < a.L && n < kMaxWords; ++i) {
      const int t = a.hyp[(size_t)hI * a.L + i];
      if (t == a.eos) break;
      if (t != a.pad) s_words[n++] = t;
    }
    s_nw = n;
    int T = 0;
    for (int k = 1; k <= 4; ++k) T += max(0, n - k + 1);
    s_T = T;
    for (int k = 0; k < 4; ++k) { s_norm[k] = 0.0; s_score[k] = 0.0; }
  }
  __syncthreads();
  const int nw = s_nw, T = s_T;
  for (int e = tid; e < T; e += kThreads) {
    int k = 1, base = 0;
    while (e >= base + (nw - k + 1)) { base += nw - k + 1; ++k; }
    const int i = e - base;
    unsigned long long key = 0;
    for (int j = 0; j < k; ++j) key |= (unsigned long long)(s_words[i + j] & 0xffff) << (16 * j);
    s_key[e] = key;
    s_ord[e] = k - 1;
  }
  __syncthreads();
  for (int e = tid; e < T; e += kThreads) {
    const unsigned long long key = s_key[e];
    int tf = 0; bool first = true;
    for (int j = 0; j < T; ++j) if (s_key[j] == key) { ++tf; if (j < e) first = false; }
    if constexpr (M == kBleu) {   // min(count_h, max over the references of count_r)
      int c = 0;
      if (first) {
        const int img = a.hyp_img[hI];
        const long k0 = b.img_key_off[img], kn = b.img_key_off[img + 1] - k0;
        const long p = lower_bound(b.keys + k0, kn, key);
        if (p < kn && b.keys[k0 + p] == key) c = min(tf, b.max_count[k0 + p]);
      }
      s_tf[e] = c;
    } else {
      s_tf[e] = first ? tf : 0;
      double v = 0.0;
      if (first) {
        const long p = lower_bound(a.df_keys, a.n_df, key);
        const double dl = (p < a.n_df && a.df_keys[p] == key) ? a.df_log[p] : 0.0;
        v = (double)tf * (a.ref_len - dl);
      }
      s_vec[e] = v;
    }
  }
  __syncthreads();
  if constexpr (M == kBleu) {
    if (tid == 0) {
      const int img = a.hyp_img[hI];
      long long st[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
      for (int e = 0; e < T; ++e) st[s_ord[e]] += s_tf[e];
      for (int k = 0; k < 4; ++k) st[4 + k] = max(0, nw - k);
      st[8] = nw;
      // the reference length l minimising (|l - testlen|, l): a tie goes to the shorter reference
      long best = -1, best_d = 0;
      for (long r = b.img_ref_off[img]; r < b.img_ref_off[img + 1]; ++r) {
        const long l = b.ref_tok_off[r + 1] - b.ref_tok_off[r], d = l > nw ? l - nw : nw - l;
        if (best < 0 || d < best_d || (d == best_d && l < best)) { best = l; best_d = d; }
      }
      st[9] = best;
      for (int i = 0; i < 10; ++i) b.stats[(size_t)img * 10 + i] = st[i];
      atomicAdd(b.hyp_count + img, 1);
    }
    return;
  }
  if (tid == 0) {
    for (int e = 0; e < T; ++e) if (s_tf[e]) s_norm[s_ord[e]] += s_vec[e] * s_vec[e];
    for (int k = 0; k < 4; ++k) s_norm[k] = sqrt(s_norm[k]);
  }
  __syncthreads();
  const int len_h = max(0, nw - 1);   // the reference counts the hypothesis' bigrams (ciderD_scorer.py:157-158)
  const int img = a.hyp_img[hI];
  const long r0 = a.img_ref_off[img], r1 = a.img_ref_off[img + 1];
  for (long r = r0; r < r1; ++r) {
    const long g0 = a.ref_ng_off[r], gn = a.ref_ng_off[r + 1] - g0;
    for (int e = tid; e < T; e += kThreads) {
      double v = 0.0;
      if (s_tf[e]) {
        const long p = lower_bound(a.ref_keys + g0, gn, s_key[e]);
        if (p < gn && a.ref_keys[g0 + p] == s_key[e]) v = a.ref_vec[g0 + p];
      }
      s_ref[e] = v;
    }
    __syncthreads();
    if (tid == 0) {
      double val[4] = {0.0, 0.0, 0.0, 0.0};
      for (int e = 0; e < T; ++e) if (s_tf[e]) val[s_ord[e]] += (M == kCiderD ? fmin(s_vec[e], s_ref[e]) : s_vec[e]) * s_ref[e];
      double pen = 1.0;
      if (M == kCiderD) {
        const double delta = (double)(len_h - a.ref_length[r]);
        pen = pow(2.718281828459045, -(delta * delta) / (2.0 * a.sigma * a.sigma));
      }
      for (int k = 0; k < 4; ++k) {
        const double nr = a.ref_norm[r * 4 + k];
        if (s_norm[k] != 0.0 && nr != 0.0) val[k] /= s_norm[k] * nr;
        if (M == kCiderD) val[k] *= pen;
        s_score[k] += val[k];
      }
    }
    __syncthreads();
  }
  if (tid == 0) {
    double s = ((s_score[0] + s_score[1]) + s_score[2]) + s_score[3];
    s /= 4.0;
    s /= (double)(r1 - r0);
    s *= 10.0;
    a.out[M == kCiderD ? hI : img] = s;
  }
}

// SCST rollout -> teacher-forcing inputs of the training step (utils/training.py:239-255, RewardCriterion utils/losses.py:10-29).
// One CTA: the token count and the mean reward are block reductions in a fixed order (bit-reproducible, no atomics), and
// inv_norm can be written by the same launch that counts.
constexpr int kTargetThreads = 1024;

__device__ __forceinline__ double scst_reward(const double* score, const double* base, int r, int S, float w) {
  double b;
  if (base != nullptr) {
    b = base[r / S];
  } else {  // mean of the image's OTHER samples (scst/scorers.py:100-106): (sum - own) / (S - 1), summed in sample order
    const int r0 = r - r % S;
    double tot = 0.0;
    for (int j = 0; j < S; ++j) tot += score[r0 + j];
    b = (tot - score[r]) / (double)(S - 1);
  }
  return (double)w * (score[r] - b);
}

template <typename T>
__device__ T block_sum(T v, T* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) red[warp] = v;
  __syncthreads();
  T s = T(0);
  if (threadIdx.x == 0) {
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
  }
  __syncthreads();
  return s;   // valid in thread 0
}

__global__ void __launch_bounds__(kTargetThreads) scst_targets_kernel(
    const int* __restrict__ seq, int R, int L, int S, const double* __restrict__ score, const double* __restrict__ base,
    float cider_weight, int bos, int pad, int* __restrict__ tokens, int* __restrict__ targets, float* __restrict__ tok_w,
    float* __restrict__ key_valid, float* __restrict__ mask_sum, float* __restrict__ inv_norm, const float* __restrict__ norm_in,
    float* __restrict__ mean_reward) {
  __shared__ long long red_i[kTargetThreads / 32];
  __shared__ double red_d[kTargetThreads / 32];
  long long count = 0;
  const long long n = (long long)R * L;
  for (long long e = threadIdx.x; e < n; e += blockDim.x) {
    const int r = (int)(e / L), t = (int)(e % L);
    const int* s = seq + (size_t)r * L;
    const int prev = t == 0 ? bos : s[t - 1];        // tokens = [BOS, s_0 .. s_{L-2}]
    const int m = (t == 0 || prev != pad) ? 1 : 0;   // RewardCriterion's mask, shifted right by one, first column 1
    tokens[e] = prev;
    targets[e] = s[t];
    key_valid[e] = prev != pad ? 1.f : 0.f;
    tok_w[e] = m ? (float)scst_reward(score, base, r, S, cider_weight) : 0.f;   // (reward -> fp32 first, like .float())
    count += m;
  }
  double rsum = 0.0;
  for (int r = threadIdx.x; r < R; r += blockDim.x) rsum += scst_reward(score, base, r, S, cider_weight);
  const long long c = block_sum(count, red_i);
  const double rs = block_sum(rsum, red_d);
  if (threadIdx.x == 0) {
    if (mask_sum) *mask_sum = (float)c;
    *inv_norm = 1.0f / (norm_in ? *norm_in : (float)c);
    if (mean_reward) *mean_reward = (float)(rs / (double)R);
  }
}

}  // namespace

extern "C" {

int sc_scst_targets(const int* seq, int R, int L, int S, const double* score, const double* base_score, float cider_weight,
                    int bos, int pad, int* tokens, int* targets, float* tok_w, float* key_valid, float* mask_sum, float* inv_norm,
                    const float* norm_in, float* mean_reward, cudaStream_t stream) {
  SC_CHECK(R > 0 && L > 0 && S > 0 && R % S == 0, SC_ERR_SHAPE, "sc_scst_targets: R=%d L=%d S=%d", R, L, S);
  SC_CHECK(base_score != nullptr || S >= 2, SC_ERR_SHAPE, "sc_scst_targets: the mean-of-others baseline needs S >= 2 samples (S=%d)", S);
  SC_CHECK(seq && score && tokens && targets && tok_w && key_valid && inv_norm, SC_ERR_SHAPE, "sc_scst_targets: null argument");
  scst_targets_kernel<<<1, kTargetThreads, 0, stream>>>(seq, R, L, S, score, base_score, cider_weight, bos, pad, tokens, targets,
                                                        tok_w, key_valid, mask_sum, inv_norm, norm_in, mean_reward);
  SC_LAUNCH_CHECK("sc_scst_targets");
  return SC_OK;
}

int sc_ciderd_score(const int* hyp, int H, int L, const int* hyp_img, int eos, int pad, const unsigned long long* df_keys,
                    const double* df_log, long n_df, double ref_len, double sigma, const long* img_ref_off, const long* ref_ng_off,
                    const unsigned long long* ref_keys, const double* ref_vec, const double* ref_norm, const int* ref_length,
                    double* out, cudaStream_t stream) {
  SC_CHECK(H > 0 && L > 0 && L <= kMaxWords, SC_ERR_SHAPE, "sc_ciderd_score: H=%d L=%d (L <= %d)", H, L, kMaxWords);
  SC_CHECK(hyp && hyp_img && img_ref_off && ref_ng_off && ref_norm && ref_length && out, SC_ERR_SHAPE, "sc_ciderd_score: null argument");
  CiderArgs a;
  a.hyp = hyp; a.L = L; a.H = H; a.hyp_img = hyp_img; a.eos = eos; a.pad = pad; a.df_keys = df_keys; a.df_log = df_log; a.n_df = n_df;
  a.ref_len = ref_len; a.sigma = sigma; a.img_ref_off = img_ref_off; a.ref_ng_off = ref_ng_off; a.ref_keys = ref_keys;
  a.ref_vec = ref_vec; a.ref_norm = ref_norm; a.ref_length = ref_length; a.out = out;
  ngram_score_kernel<kCiderD><<<H, kThreads, 0, stream>>>(a, BleuArgs{}, 0);
  SC_LAUNCH_CHECK("sc_ciderd_score");
  return SC_OK;
}

int sc_cider_score(const int* hyp, int H, int L, const int* hyp_img, int n_images, int eos, int pad, const unsigned long long* df_keys,
                   const double* df_log, long n_df, double ref_len, const long* img_ref_off, const long* ref_ng_off,
                   const unsigned long long* ref_keys, const double* ref_vec, const double* ref_norm, double* out, cudaStream_t stream) {
  SC_CHECK(H > 0 && L > 0 && L <= kMaxWords && n_images > 0, SC_ERR_SHAPE, "sc_cider_score: H=%d L=%d (L <= %d) n_images=%d", H, L,
           kMaxWords, n_images);
  SC_CHECK(hyp && hyp_img && img_ref_off && ref_ng_off && ref_norm && out, SC_ERR_SHAPE, "sc_cider_score: null argument");
  CiderArgs a = {};
  a.hyp = hyp; a.L = L; a.H = H; a.hyp_img = hyp_img; a.eos = eos; a.pad = pad; a.df_keys = df_keys; a.df_log = df_log; a.n_df = n_df;
  a.ref_len = ref_len; a.img_ref_off = img_ref_off; a.ref_ng_off = ref_ng_off; a.ref_keys = ref_keys; a.ref_vec = ref_vec;
  a.ref_norm = ref_norm; a.out = out;
  ngram_score_kernel<kCider><<<H, kThreads, 0, stream>>>(a, BleuArgs{}, n_images);
  SC_LAUNCH_CHECK("sc_cider_score");
  return SC_OK;
}

int sc_bleu_stats(const int* hyp, int H, int L, const int* hyp_img, int n_images, int eos, int pad, const long* img_key_off,
                  const unsigned long long* keys, const int* max_count, const long* img_ref_off, const long* ref_tok_off,
                  long long* stats, int* hyp_count, int* bad_index, cudaStream_t stream) {
  SC_CHECK(H > 0 && L > 0 && L <= kMaxWords && n_images > 0, SC_ERR_SHAPE, "sc_bleu_stats: H=%d L=%d (L <= %d) n_images=%d", H, L,
           kMaxWords, n_images);
  SC_CHECK(hyp && hyp_img && img_key_off && keys && max_count && img_ref_off && ref_tok_off && stats && hyp_count && bad_index,
           SC_ERR_SHAPE, "sc_bleu_stats: null argument");
  CiderArgs a = {};
  a.hyp = hyp; a.L = L; a.H = H; a.hyp_img = hyp_img; a.eos = eos; a.pad = pad;
  const BleuArgs b = {img_key_off, keys, max_count, img_ref_off, ref_tok_off, stats, hyp_count, bad_index};
  ngram_score_kernel<kBleu><<<H, kThreads, 0, stream>>>(a, b, n_images);
  SC_LAUNCH_CHECK("sc_bleu_stats");
  return SC_OK;
}

}  // extern "C"
