"""coco-caption validation metrics, CPU tier: the oracle (oracle/caption_metrics_oracle.py) on hand-worked BLEU / ROUGE-L / CIDEr
cases, its CIDEr with CIDEr-D's clip and penalty switched on against the golden of the imported CIDEr-D scorer, and
``encode_refs``."""
import math
import os

import numpy as np
import pytest

from oracle import caption_metrics_oracle as M
from oracle import cider_oracle as C

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ciderd.npz")
A, B, CC, D, E, X = 5, 6, 7, 8, 9, 10    # word ids


def test_bleu_clips_counts_to_the_reference_max():
    # "the the the the" vs "the cat": unigram "the" counted min(4, 1) = 1 times
    comps = M.bleu_cook_test([A, A, A, A], M.bleu_cook_refs([[A, B]]))
    assert comps == {"reflen": 2, "testlen": 4, "guess": [4, 3, 2, 1], "correct": [1, 0, 0, 0]}
    # the max is per reference, not summed over references: two references with one "the" each still allow 1
    assert M.bleu_cook_test([A, A, A, A], M.bleu_cook_refs([[A, B], [B, A]]))["correct"][0] == 1
    assert M.bleu_cook_test([A, A, A, A], M.bleu_cook_refs([[A, B], [A, A, B]]))["correct"][0] == 2
    bleus, per = M.bleu([[A, A, A, A]], [[[A, B]]])
    assert bleus[0] == pytest.approx(0.25, rel=1e-9) and per[0][0] == bleus[0]   # testlen >= reflen: no brevity penalty


def test_bleu_brevity_penalty():
    # "a b" vs "a b c d": every unigram / bigram matches, ratio 2/4 -> BLEU_1 = exp(1 - 2) = 1/e
    bleus, per = M.bleu([[A, B]], [[[A, B, CC, D]]])
    assert bleus[0] == pytest.approx(math.exp(-1.0), rel=1e-8)   # (small = 1e-9 in the precision's denominator)
    assert bleus[1] == pytest.approx(math.exp(-1.0), rel=1e-8)
    assert bleus[2] == pytest.approx(0.01 * math.exp(-1.0), rel=1e-6)   # no trigram: p3 = tiny / small = 1e-6, cube root


def test_bleu_closest_reference_length_tie_goes_to_the_shorter():
    for refs in ([[A, B], [A, B, CC, D]], [[A, B, CC, D], [A, B]]):
        assert M.bleu_cook_test([A, B, CC], M.bleu_cook_refs(refs))["reflen"] == 2
    assert M.bleu_cook_test([A, B, CC], M.bleu_cook_refs([[A], [A, B, CC, D]]))["reflen"] == 4


def test_empty_hypothesis_scores_zero():
    refs = [[[A, B, CC]], [[D, E]]]
    scores, per = M.evaluate([[], [D, E]], refs)
    assert per[0].tolist() == [0.0] * 6
    assert M.bleu_cook_test([], M.bleu_cook_refs(refs[0])) == {"reflen": 3, "testlen": 0, "guess": [0, 0, 0, 0],
                                                               "correct": [0, 0, 0, 0]}
    assert M.rouge_l([], [[A]]) == 0.0


def test_rouge_l_hand_worked():
    assert M.my_lcs([A, B, CC], [A, X, CC, D, E]) == 2
    assert M.my_lcs([A, CC, E, D], [A, B, CC, D]) == 3
    # P = 2/3, R = 2/5, beta^2 = 1.44: 2.44 * (4/15) / (2/5 + 0.96) = 122/255
    assert M.rouge_l([A, B, CC], [[A, X, CC, D, E]]) == pytest.approx(122 / 255, rel=1e-14)
    # P and R are maxima over the references, taken separately
    assert M.rouge_l([A, B], [[A, B, CC, D, E, X], [A, X]]) == pytest.approx(2.44 * 1.0 * (1 / 2) / (1 / 2 + 1.44), rel=1e-14)


def test_cider_without_the_clip_differs_from_cider_d():
    # two images -> idf log(2) for every reference n-gram; hypothesis "a a" for references "a b":
    # unigram cosine = (2 log2 . log2) / (2 log2 . sqrt(2) log2) = 1/sqrt(2) unclipped, 1/(2 sqrt(2)) with CIDEr-D's clip;
    # no bigram in common, no 3- or 4-grams; both have one bigram, so the length penalty is 1
    refs = [[[A, B]], [[CC, D]]]
    hyps = [[A, A], [CC, D]]
    df = C.corpus_document_frequency(refs)
    ref_len = np.log(2.0)
    got = M.cider_scores(hyps, refs, df, ref_len)
    assert got[0] == pytest.approx(10 / (4 * math.sqrt(2)), rel=1e-14)
    assert got[1] == pytest.approx(5.0, rel=1e-14)             # exact copy: unigram and bigram cosine 1
    clipped = M.cider_scores(hyps, refs, df, ref_len, clip=True, penalty=True)
    assert clipped[0] == pytest.approx(10 / (8 * math.sqrt(2)), rel=1e-14)
    assert np.array_equal(M.cider(hyps, refs), got)


def test_cider_with_clip_and_penalty_is_the_ciderd_oracle_on_the_golden():
    z = np.load(GOLDEN)
    unpad = lambda a: [[int(x) for x in r if x >= 0] for r in a]
    refs_flat, hyps = unpad(z["refs"]), unpad(z["hyps"])
    refs, o = [], 0
    for c in z["ref_count"]:
        refs.append(refs_flat[o: o + int(c)])
        o += int(c)
    ns = len(hyps) // len(refs)
    rr = [refs[i // ns] for i in range(len(hyps))]
    df = C.corpus_document_frequency(rr)
    got = M.cider_scores(hyps, rr, df, np.log(float(len(rr))), clip=True, penalty=True)
    assert np.array_equal(got, C.ciderd(hyps, rr, df, np.log(float(len(rr)))))
    assert np.array_equal(got, z["corpus_scores"])


def test_evaluate_per_image_columns():
    refs = [[[A, B, CC, D], [A, B, E]], [[D, E, X]], [[CC, CC, A]]]
    hyps = [[A, B, CC], [D, E, X], [A]]
    scores, per = M.evaluate(hyps, refs)
    assert list(scores) == list(M.METRICS) and per.shape == (3, 6) and per.dtype == np.float64
    assert scores["ROUGE_L"] == pytest.approx(per[:, 4].mean(), rel=1e-15)
    assert scores["CIDEr"] == pytest.approx(per[:, 5].mean(), rel=1e-15)
    assert per[1, 4] == 1.0 and per[1, 0] == pytest.approx(1.0, rel=1e-9)


def test_encode_refs_gives_out_of_vocabulary_words_fresh_ids():
    from sparse_caption_b200.metrics import encode_refs
    vocab = {"<pad>": 0, "<unk>": 1, "<bos>": 2, "<eos>": 3, "a": 4, "dog": 5, "runs": 6}
    got = encode_refs([["a dog runs", "a zebra runs"], ["a zebra", "an okapi dog"]], vocab)
    assert got == [[[4, 5, 6], [4, 7, 6]], [[4, 7], [8, 9, 5]]]
    assert all(w != vocab["<unk>"] for img in got for ref in img for w in ref)
    with pytest.raises(ValueError, match="65536"):
        encode_refs([[" ".join(f"w{i}" for i in range(70000))]], vocab)
