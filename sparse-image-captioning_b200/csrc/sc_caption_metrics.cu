// coco-caption validation metrics on word ids, the part that is not n-gram counting (sc_cider.cu computes BLEU's statistics and
// CIDEr): ROUGE-L (pycocoevalcap rouge/rouge.py) and the corpus / per-image numbers of a split (bleu/bleu_scorer.py
// compute_score, the means of coco_caption/eval.py:15-86).  Kept out of sc_cider.cu so that its pow / exp calls do not change
// the inlining, and so the code, of the CIDEr-D kernel there.
#include "sc_common.cuh"

namespace {

constexpr int kMaxWords = 64;

// ROUGE-L of rouge.py (beta = 1.2): one warp per hypothesis, the exact LCS with every reference by the bit-parallel algorithm of
// Allison-Dix / Hyyro over the <= 64 hypothesis positions (bit i = word i; lane l holds words l and l + 32).  Per reference
// token t: M = positions holding t (two ballots), V = (V + (V & M)) | (V & ~M); LCS = the zero bits of V below |h|.
constexpr int kRougeWarps = 4;

__global__ void __launch_bounds__(kRougeWarps * 32) rouge_l_kernel(const int* __restrict__ hyp, int H, int L,
                                                                   const int* __restrict__ hyp_img, int n_img, int eos, int pad,
                                                                   const long* __restrict__ img_ref_off,
                                                                   const long* __restrict__ ref_tok_off,
                                                                   const int* __restrict__ ref_tok, double* __restrict__ out) {
  __shared__ int s_words[kRougeWarps][kMaxWords];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int h = blockIdx.x * kRougeWarps + w;
  if (h >= H) return;
  const int img = hyp_img[h];
  if (img < 0 || img >= n_img) return;
  // compact the caption: positions before the first <eos>, pads dropped (L <= 64)
  const int* row = hyp + (size_t)h * L;
  const int t0 = lane < L ? row[lane] : eos, t1 = lane + 32 < L ? row[lane + 32] : eos;
  const unsigned e0 = __ballot_sync(0xffffffffu, t0 == eos), e1 = __ballot_sync(0xffffffffu, t1 == eos);
  const int first_eos = e0 ? __ffs(e0) - 1 : (e1 ? 32 + __ffs(e1) - 1 : 64);
  const bool k0 = lane < first_eos && t0 != pad, k1 = lane + 32 < first_eos && t1 != pad;
  const unsigned m0 = __ballot_sync(0xffffffffu, k0), m1 = __ballot_sync(0xffffffffu, k1);
  const unsigned below = (1u << lane) - 1u;
  if (k0) s_words[w][__popc(m0 & below)] = t0;
  if (k1) s_words[w][__popc(m0) + __popc(m1 & below)] = t1;
  const int nw = __popc(m0) + __popc(m1);
  __syncwarp();
  const int w0 = lane < nw ? s_words[w][lane] : -1, w1 = lane + 32 < nw ? s_words[w][lane + 32] : -1;   // ids are > 0
  const unsigned long long used = nw == 64 ? ~0ull : (1ull << nw) - 1ull;
  double P = 0.0, R = 0.0;
  for (long r = img_ref_off[img]; r < img_ref_off[img + 1]; ++r) {
    const long o0 = ref_tok_off[r], n = ref_tok_off[r + 1] - o0;
    unsigned long long V = ~0ull;
    for (long c = 0; c < n; c += 32) {
      const int mine = c + lane < n ? ref_tok[o0 + c + lane] : 0;
      const int m = n - c < 32 ? (int)(n - c) : 32;
      for (int j = 0; j < m; ++j) {
        const int t = __shfl_sync(0xffffffffu, mine, j);
        const unsigned long long M = (unsigned long long)__ballot_sync(0xffffffffu, w0 == t) |
                                     ((unsigned long long)__ballot_sync(0xffffffffu, w1 == t) << 32);
        V = (V + (V & M)) | (V & ~M);
      }
    }
    const int lcs = nw - __popcll(V & used);
    // rouge.py: prec = lcs / |h|, rec = lcs / |r| (an empty side has lcs 0 and contributes 0)
    if (nw > 0) P = fmax(P, (double)lcs / (double)nw);
    if (n > 0) R = fmax(R, (double)lcs / (double)n);
  }
  if (lane == 0) {
    const double b2 = __dmul_rn(1.2, 1.2);   // self.beta ** 2
    double score = 0.0;
    if (P != 0.0 && R != 0.0) score = __dmul_rn(__dmul_rn(__dadd_rn(1.0, b2), P), R) / __dadd_rn(R, __dmul_rn(b2, P));
    out[img] = score;
  }
}

// Corpus and per-image numbers of one split in one CTA, in a fixed order (bitwise reproducible): BLEU from the int64 sums of
// the statistics (bleu_scorer.py compute_score: tiny = 1e-15, small = 1e-9, cumulative product ^ 1/k, brevity penalty when
// testlen < reflen), per-image BLEU_k (bleu_list) from one image's statistics by the same formula, means of ROUGE-L and CIDEr.
constexpr int kReduceThreads = 256;

__device__ __forceinline__ void bleu_from_stats(const long long* st, double* bleus) {
  const double tiny = 1e-15, small = 1e-9;
  double bleu = 1.0;
  for (int k = 0; k < 4; ++k) {
    bleu = __dmul_rn(bleu, __dadd_rn((double)st[k], tiny) / __dadd_rn((double)st[4 + k], small));
    bleus[k] = pow(bleu, 1.0 / (double)(k + 1));
  }
  const double ratio = __dadd_rn((double)st[8], tiny) / __dadd_rn((double)st[9], small);
  if (ratio < 1.0) {
    const double bp = exp(1.0 - 1.0 / ratio);
    for (int k = 0; k < 4; ++k) bleus[k] = __dmul_rn(bleus[k], bp);
  }
}

__global__ void __launch_bounds__(kReduceThreads) caption_metrics_reduce_kernel(
    const long long* __restrict__ stats, const double* __restrict__ rouge, const double* __restrict__ cider,
    const int* __restrict__ hyp_count, const int* __restrict__ bad_index, int n_img, double* __restrict__ out) {
  __shared__ long long s_int[12][kReduceThreads];
  __shared__ double s_dbl[2][kReduceThreads];
  long long sum[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, missing = 0, repeated = 0;
  double rs = 0.0, cs = 0.0;
  double* per_img = out + 9;
  for (int i = threadIdx.x; i < n_img; i += kReduceThreads) {
    const long long* st = stats + (size_t)i * 10;
    for (int j = 0; j < 10; ++j) sum[j] += st[j];
    double bl[4];
    bleu_from_stats(st, bl);
    for (int k = 0; k < 4; ++k) per_img[(size_t)i * 6 + k] = bl[k];
    per_img[(size_t)i * 6 + 4] = rouge[i];
    per_img[(size_t)i * 6 + 5] = cider[i];
    rs += rouge[i];
    cs += cider[i];
    missing += hyp_count[i] == 0;
    repeated += hyp_count[i] > 1;
  }
  const int t = threadIdx.x;
  for (int j = 0; j < 10; ++j) s_int[j][t] = sum[j];
  s_int[10][t] = missing;
  s_int[11][t] = repeated;
  s_dbl[0][t] = rs;
  s_dbl[1][t] = cs;
  __syncthreads();
  if (t == 0) {   // partials in thread order
    for (int i = 1; i < kReduceThreads; ++i) {
      for (int j = 0; j < 10; ++j) sum[j] += s_int[j][i];
      missing += s_int[10][i];
      repeated += s_int[11][i];
      rs += s_dbl[0][i];
      cs += s_dbl[1][i];
    }
    bleu_from_stats(sum, out);
    out[4] = rs / (double)n_img;
    out[5] = cs / (double)n_img;
    out[6] = (double)missing;
    out[7] = (double)repeated;
    out[8] = (double)*bad_index;
  }
}

}  // namespace

extern "C" {

int sc_rouge_l(const int* hyp, int H, int L, const int* hyp_img, int n_images, int eos, int pad, const long* img_ref_off,
               const long* ref_tok_off, const int* ref_tok, double* out, cudaStream_t stream) {
  SC_CHECK(H > 0 && L > 0 && L <= kMaxWords && n_images > 0, SC_ERR_SHAPE, "sc_rouge_l: H=%d L=%d (L <= %d) n_images=%d", H, L,
           kMaxWords, n_images);
  SC_CHECK(hyp && hyp_img && img_ref_off && ref_tok_off && ref_tok && out, SC_ERR_SHAPE, "sc_rouge_l: null argument");
  rouge_l_kernel<<<(H + kRougeWarps - 1) / kRougeWarps, kRougeWarps * 32, 0, stream>>>(hyp, H, L, hyp_img, n_images, eos, pad,
                                                                                      img_ref_off, ref_tok_off, ref_tok, out);
  SC_LAUNCH_CHECK("sc_rouge_l");
  return SC_OK;
}

int sc_caption_metrics_reduce(const long long* bleu_stats, const double* rouge, const double* cider, const int* hyp_count,
                              const int* bad_index, int n_images, double* out, cudaStream_t stream) {
  SC_CHECK(n_images > 0, SC_ERR_SHAPE, "sc_caption_metrics_reduce: n_images=%d", n_images);
  SC_CHECK(bleu_stats && rouge && cider && hyp_count && bad_index && out, SC_ERR_SHAPE, "sc_caption_metrics_reduce: null argument");
  caption_metrics_reduce_kernel<<<1, kReduceThreads, 0, stream>>>(bleu_stats, rouge, cider, hyp_count, bad_index, n_images, out);
  SC_LAUNCH_CHECK("sc_caption_metrics_reduce");
  return SC_OK;
}

}  // extern "C"
