"""CIDEr-D reward on the device - the step after the path for SCST (SURVEY.md section 8f.4).

Drop-in for the reward part of ``TrainingModule.compute_scst_loss`` (utils/training.py:239-252): the reference detokenises
B x (samples + 1) rollouts to strings and scores them with ``CaptionScorer`` (scst/scorers.py:47-114 -> CiderD,
scst/cider/pyciderevalcap/ciderD/ciderD_scorer.py) in Python; here the rollouts stay on the device as word ids and
``sc_ciderd_score`` returns the scores there, so rollout -> reward -> teacher-forced backward never leaves the GPU.

The static parts are prepared once on the host with the reference's own arithmetic (Python floats / numpy float64): the
document-frequency table (``coco-train-words.p`` in the reference, or "corpus" mode) and the tf-idf vector, norm and length of
every reference caption.
"""
import math
from collections import defaultdict
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import lib

Ngram = Tuple[int, ...]


def _key(ngram: Sequence[int]) -> int:
    k = 0
    for j, w in enumerate(ngram):
        assert 0 < int(w) < 65536, "word ids must be in [1, 65535] (16 bits per n-gram slot)"
        k |= int(w) << (16 * j)
    return k


def _precook(words: Sequence[int], n: int = 4) -> Dict[Ngram, int]:
    counts: Dict[Ngram, int] = defaultdict(int)
    for k in range(1, n + 1):
        for i in range(len(words) - k + 1):
            counts[tuple(int(w) for w in words[i: i + k])] += 1
    return counts


class CiderD:
    """``df``: {n-gram of word ids: document frequency}; ``n_docs``: number of documents behind it (``ref_len`` = log of it).
    ``CiderD.from_corpus(refs)`` computes both from the given references (the scorer's "corpus" mode)."""

    def __init__(self, df: Dict[Ngram, float], n_docs: float, *, device="cuda", sigma: float = 6.0, eos_id: int = 3, pad_id: int = 0):
        self.dev = lib.resolve_device(device)
        self.sigma, self.eos, self.pad = float(sigma), int(eos_id), int(pad_id)
        self.df = df
        self.ref_len = float(np.log(float(n_docs)))
        items = sorted((_key(ng), float(np.log(max(1.0, c)))) for ng, c in df.items())
        self.df_keys = torch.from_numpy(np.array([k for k, _ in items] or [0], dtype=np.uint64).view(np.int64)).to(self.dev)
        self.df_log = torch.tensor([v for _, v in items] or [0.0], dtype=torch.float64, device=self.dev)
        self.n_df = len(items)
        self._refs = None

    @classmethod
    def from_corpus(cls, refs_per_image: Sequence[Sequence[Sequence[int]]], **kw):
        df: Dict[Ngram, float] = defaultdict(float)
        for refs in refs_per_image:
            for ng in set(ng for ref in refs for ng in _precook(ref)):
                df[ng] += 1
        self = cls(df, float(len(refs_per_image)), **kw)
        self.set_refs(refs_per_image)
        return self

    def set_refs(self, refs_per_image: Sequence[Sequence[Sequence[int]]]) -> None:
        """tf-idf vectors / norms / lengths of the reference captions (counts2vec, ciderD_scorer.py:134-160), per image: of a batch, or
        of a whole split once (then ``score`` / ``scst_reward`` / ``scst_step`` take dataset image indices)."""
        img_off, ng_off, keys, vecs, norms, lens = [0], [0], [], [], [], []
        for refs in refs_per_image:
            for ref in refs:
                norm = [0.0] * 4
                length = 0
                ent = []
                for ng, tf in _precook(ref).items():
                    d = np.log(max(1.0, self.df.get(ng, 0.0)))
                    v = float(tf) * (self.ref_len - d)
                    norm[len(ng) - 1] += pow(v, 2)
                    if len(ng) == 2:
                        length += tf
                    ent.append((_key(ng), v))
                ent.sort()
                keys += [k for k, _ in ent]
                vecs += [v for _, v in ent]
                norms.append([float(np.sqrt(x)) for x in norm])
                lens.append(length)
                ng_off.append(len(keys))
            img_off.append(len(lens))
        dev = self.dev
        self._refs = dict(
            img_off=torch.tensor(img_off, dtype=torch.int64, device=dev), ng_off=torch.tensor(ng_off, dtype=torch.int64, device=dev),
            keys=torch.from_numpy(np.array(keys or [0], dtype=np.uint64).view(np.int64)).to(dev),
            vec=torch.tensor(vecs or [0.0], dtype=torch.float64, device=dev),
            norm=torch.tensor(norms, dtype=torch.float64, device=dev).reshape(-1, 4).contiguous(),
            length=torch.tensor(lens, dtype=torch.int32, device=dev), n_images=len(refs_per_image))

    def score(self, hyp: torch.Tensor, hyp_image: torch.Tensor) -> torch.Tensor:
        """hyp int [H, L] word ids on the device, hyp_image int [H] (index into the current references) -> float64 [H]."""
        assert self._refs is not None, "call set_refs() with the batch's reference captions first"
        if not hyp.is_cuda:
            raise RuntimeError("CiderD.score runs on CUDA tensors only (there is no CPU fallback)")
        H, L = hyp.shape
        h = hyp.to(torch.int32).contiguous()
        hi = hyp_image.to(self.dev, torch.int32).contiguous()
        out = torch.empty(H, dtype=torch.float64, device=self.dev)
        r = self._refs
        lib.call("sc_ciderd_score", h, H, L, hi, self.eos, self.pad, self.df_keys, self.df_log, self.n_df, self.ref_len, self.sigma,
                 r["img_off"], r["ng_off"], r["keys"], r["vec"], r["norm"], r["length"], out)
        return out

    def scst_reward(self, sample_seq: torch.Tensor, baseline_seq: Optional[torch.Tensor] = None, cider_weight: float = 1.0,
                    image_ids: Optional[torch.Tensor] = None):
        """CaptionScorer.__call__ (scorers.py:47-114): ``sample_seq`` [B, n, L] rollouts, ``baseline_seq`` [B, 1, L] greedy captions or
        None (then each sample's baseline is the mean score of the image's OTHER samples).  ``image_ids`` [B]: the images' indices
        into the references given to ``set_refs`` (default 0 .. B-1): ``set_refs`` can then take a whole split once instead of
        every batch.  Returns (sc_sample, sc_baseline), float64 [B * n] on the device; the SCST reward is their difference
        (training.py:252)."""
        B, n, L = sample_seq.shape
        ids = torch.arange(B, device=self.dev) if image_ids is None else torch.as_tensor(image_ids).to(self.dev)
        img = ids.repeat_interleave(n)
        sc_sample = self.score(sample_seq.reshape(B * n, L), img) * cider_weight
        if baseline_seq is not None:
            sc_b = self.score(baseline_seq.reshape(B, -1)[:, :L], ids) * cider_weight
            return sc_sample, sc_b.repeat_interleave(n)
        tot = sc_sample.view(B, n).sum(-1)
        return sc_sample, (tot.repeat_interleave(n) - sc_sample) / (n - 1)
