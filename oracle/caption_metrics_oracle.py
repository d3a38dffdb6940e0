"""CPU oracle for the coco-caption validation metrics BLEU-1..4, ROUGE-L and CIDEr.  TEST INFRASTRUCTURE ONLY (see ort_oracle.py).

Restates pycocoevalcap ``bleu/bleu_scorer.py`` (precook, cook_refs, cook_test with option "closest", compute_score),
``rouge/rouge.py`` (my_lcs, Rouge.calc_score, beta = 1.2) and ``cider/cider_scorer.py`` (compute_doc_freq, compute_cider) as
called by ``coco_caption/eval.py:15-86``, in Python floats on captions given as lists of word ids instead of whitespace-split
strings.  CIDEr reuses ``cider_oracle`` (CIDEr-D's counts2vec / precook / document frequency): CIDEr is CIDEr-D without the
clip of the hypothesis tf-idf and without the Gaussian length penalty, and with both switched on ``cider`` equals
``cider_oracle.ciderd``, which is pinned to the imported reference scorer by tests/golden/ciderd.npz.
BLEU and ROUGE-L are pinned by hand-worked cases (tests/test_caption_metrics_cpu.py).
"""
import math
from collections import defaultdict
from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import cider_oracle as C

Ngram = Tuple[int, ...]
METRICS = ("Bleu_1", "Bleu_2", "Bleu_3", "Bleu_4", "ROUGE_L", "CIDEr")


# ---- BLEU (bleu_scorer.py) ----
def bleu_precook(words: Sequence[int], n: int = 4):
    counts: Dict[Ngram, int] = defaultdict(int)
    for k in range(1, n + 1):
        for i in range(len(words) - k + 1):
            counts[tuple(words[i: i + k])] += 1
    return len(words), counts


def bleu_cook_refs(refs: Sequence[Sequence[int]], n: int = 4):
    reflen, maxcounts = [], {}
    for ref in refs:
        rl, counts = bleu_precook(ref, n)
        reflen.append(rl)
        for ngram, count in counts.items():
            maxcounts[ngram] = max(maxcounts.get(ngram, 0), count)
    return reflen, maxcounts


def bleu_cook_test(test: Sequence[int], crefs, n: int = 4) -> dict:
    """cook_test with eff="closest": the reference length l minimising (|l - testlen|, l)."""
    testlen, counts = bleu_precook(test, n)
    reflen, refmaxcounts = crefs
    result = {"reflen": min((abs(l - testlen), l) for l in reflen)[1], "testlen": testlen,
              "guess": [max(0, testlen - k + 1) for k in range(1, n + 1)], "correct": [0] * n}
    for ngram, count in counts.items():
        result["correct"][len(ngram) - 1] += min(refmaxcounts.get(ngram, 0), count)
    return result


def bleu(hyps: Sequence[Sequence[int]], refs: Sequence[Sequence[Sequence[int]]], n: int = 4):
    """BleuScorer.compute_score(option="closest"): (corpus [Bleu_1..n], per image [n][images] (bleu_list))."""
    small, tiny = 1e-9, 1e-15
    bleu_list: List[List[float]] = [[] for _ in range(n)]
    testlen_t = reflen_t = 0
    totalcomps = {"guess": [0] * n, "correct": [0] * n}
    for test, rs in zip(hyps, refs):
        comps = bleu_cook_test(test, bleu_cook_refs(rs, n), n)
        testlen, reflen = comps["testlen"], comps["reflen"]
        testlen_t += testlen
        reflen_t += reflen
        for key in ("guess", "correct"):
            for k in range(n):
                totalcomps[key][k] += comps[key][k]
        b = 1.0
        for k in range(n):
            b *= (float(comps["correct"][k]) + tiny) / (float(comps["guess"][k]) + small)
            bleu_list[k].append(b ** (1.0 / (k + 1)))
        ratio = (testlen + tiny) / (reflen + small)
        if ratio < 1:
            for k in range(n):
                bleu_list[k][-1] *= math.exp(1 - 1 / ratio)
    bleus = []
    b = 1.0
    for k in range(n):
        b *= float(totalcomps["correct"][k] + tiny) / (totalcomps["guess"][k] + small)
        bleus.append(b ** (1.0 / (k + 1)))
    ratio = (testlen_t + tiny) / (reflen_t + small)
    if ratio < 1:
        for k in range(n):
            bleus[k] *= math.exp(1 - 1 / ratio)
    return bleus, bleu_list


# ---- ROUGE-L (rouge.py) ----
def my_lcs(string: Sequence[int], sub: Sequence[int]) -> int:
    if len(string) < len(sub):
        sub, string = string, sub
    lengths = [[0 for _ in range(0, len(sub) + 1)] for _ in range(0, len(string) + 1)]
    for j in range(1, len(sub) + 1):
        for i in range(1, len(string) + 1):
            if string[i - 1] == sub[j - 1]:
                lengths[i][j] = lengths[i - 1][j - 1] + 1
            else:
                lengths[i][j] = max(lengths[i - 1][j], lengths[i][j - 1])
    return lengths[len(string)][len(sub)]


def rouge_l(candidate: Sequence[int], refs: Sequence[Sequence[int]], beta: float = 1.2) -> float:
    """Rouge.calc_score.  The reference splits strings with split(" "), so an empty caption is one empty token that matches
    nothing: its precision (or recall) is 0, and an empty hypothesis scores 0."""
    if len(candidate) == 0:
        return 0.0
    prec, rec = [], []
    for reference in refs:
        lcs = my_lcs(reference, candidate)
        prec.append(lcs / float(len(candidate)))
        rec.append(lcs / float(len(reference)) if len(reference) else 0.0)
    prec_max, rec_max = max(prec), max(rec)
    if prec_max != 0 and rec_max != 0:
        return ((1 + beta ** 2) * prec_max * rec_max) / float(rec_max + beta ** 2 * prec_max)
    return 0.0


# ---- CIDEr (cider_scorer.py) on CIDEr-D's pieces ----
def sim(vec_h, vec_r, norm_h, norm_r, len_h, len_r, n: int = 4, sigma: float = 6.0, clip: bool = False, penalty: bool = False):
    """cider_scorer.py sim (clip = penalty = False) or ciderD_scorer.py sim (both True)."""
    delta = float(len_h - len_r)
    val = np.array([0.0 for _ in range(n)])
    for k in range(n):
        for ngram in vec_h[k]:
            h, r = vec_h[k][ngram], vec_r[k].get(ngram, 0.0)
            val[k] += (min(h, r) if clip else h) * r
        if norm_h[k] != 0 and norm_r[k] != 0:
            val[k] /= norm_h[k] * norm_r[k]
        if penalty:
            val[k] *= np.e ** (-(delta ** 2) / (2 * sigma ** 2))
    return val


def cider_scores(hyps, refs, df, ref_len, n: int = 4, sigma: float = 6.0, clip: bool = False, penalty: bool = False) -> np.ndarray:
    """compute_cider: one score per (hypothesis, reference set) pair."""
    scores = []
    for test, rs in zip(hyps, refs):
        vec, norm, length = C.counts2vec(C.precook(test, n), df, ref_len, n)
        score = np.array([0.0 for _ in range(n)])
        for ref in rs:
            vr, nr, lr = C.counts2vec(C.precook(ref, n), df, ref_len, n)
            score += sim(vec, vr, norm, nr, length, lr, n, sigma, clip, penalty)
        s = np.mean(score)
        s /= len(rs)
        s *= 10.0
        scores.append(s)
    return np.array(scores)


def cider(hyps, refs) -> np.ndarray:
    """Cider.compute_score: document frequencies from the evaluated images' references, ref_len = log(#images)."""
    return cider_scores(hyps, refs, C.corpus_document_frequency(refs), np.log(float(len(refs))))


def evaluate(hyps: Sequence[Sequence[int]], refs: Sequence[Sequence[Sequence[int]]]):
    """COCOEvalCap.evaluate restricted to BLEU, ROUGE-L and CIDEr: ({metric: corpus score}, per image float64 [n, 6])."""
    bleus, bleu_list = bleu(hyps, refs)
    rouge = np.array([rouge_l(h, rs) for h, rs in zip(hyps, refs)])
    cid = cider(hyps, refs)
    scores = dict(zip(METRICS, bleus + [float(np.mean(rouge)), float(np.mean(cid))]))
    per_image = np.stack([np.array(b) for b in bleu_list] + [rouge, cid], 1)
    return scores, per_image
