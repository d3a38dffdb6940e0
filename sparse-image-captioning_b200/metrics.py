"""coco-caption validation scores on the device: BLEU-1..4, ROUGE-L and CIDEr of ``eval_on_split`` (utils/training.py:257-327,
coco_caption/eval.py:15-86) computed on the word ids the engine returns, without detokenising the captions.

METEOR, SPICE and the PTB tokenizer (Java) are not computed; the references arrive already tokenised (``encode_refs``).
The static parts are prepared once per split on the host with the reference's own arithmetic: BLEU's per-image max n-gram
counts (bleu_scorer.py cook_refs), the reference token arrays for ROUGE-L, and a ``CiderD.from_corpus`` for CIDEr (document
frequencies from this split's references, ref_len = log(#images), as cider_scorer.py computes them).
"""
from typing import Dict, List, Mapping, Sequence, Tuple

import numpy as np
import torch

from . import lib
from .cider import CiderD, _key, _precook

METRICS = ("Bleu_1", "Bleu_2", "Bleu_3", "Bleu_4", "ROUGE_L", "CIDEr")


def encode_refs(ref_token_lists: Sequence[Sequence[str]], word_to_id: Mapping[str, int]) -> List[List[List[int]]]:
    """Tokenised reference captions (per image, a list of space-separated strings) -> word ids for ``CaptionMetrics.set_refs``.
    A word outside the model vocabulary gets a fresh id at or above the vocabulary size (the same id wherever it occurs), never
    <unk>: coco-caption compares words, so a hypothesis <unk> must not match it."""
    next_id = max(word_to_id.values()) + 1
    fresh: Dict[str, int] = {}
    out = []
    for refs in ref_token_lists:
        img = []
        for ref in refs:
            ids = []
            for w in ref.split():
                if w in word_to_id:
                    ids.append(int(word_to_id[w]))
                else:
                    if w not in fresh:
                        fresh[w] = next_id + len(fresh)
                    ids.append(fresh[w])
            img.append(ids)
        out.append(img)
    if next_id + len(fresh) > 65536:
        raise ValueError(f"{len(fresh)} out-of-vocabulary reference words do not fit word ids below 65536")
    return out


class CaptionMetrics:
    """Accumulates one hypothesis per image of a split on the device and returns coco-caption's scores.

    ``set_refs(refs_per_image)`` once per split (word ids, see ``encode_refs``); per batch ``add(seq_words, image_idx)`` with the
    device word ids [H, L <= 64] (ids before the first ``eos_id``, ``pad_id`` dropped) and each hypothesis' index into the split;
    ``compute()`` once: ({"Bleu_1" .. "CIDEr"}, per-image float64 [n_images, 6] in that column order)."""

    def __init__(self, eos_id: int = 3, pad_id: int = 0, device="cuda"):
        self.dev = lib.resolve_device(device)
        self.eos, self.pad = int(eos_id), int(pad_id)
        self.n_images = 0

    def set_refs(self, refs_per_image: Sequence[Sequence[Sequence[int]]]) -> None:
        n = len(refs_per_image)
        if n == 0:
            raise ValueError("set_refs needs at least one image")
        if any(len(refs) == 0 for refs in refs_per_image):
            raise ValueError("every image needs at least one reference caption")
        key_off, keys, max_count, img_ref_off, tok_off, toks = [0], [], [], [0], [0], []
        for refs in refs_per_image:
            mc: Dict[int, int] = {}
            for ref in refs:
                for ng, c in _precook(ref).items():
                    k = _key(ng)
                    mc[k] = max(mc.get(k, 0), c)
                toks += [int(w) for w in ref]
                tok_off.append(len(toks))
            for k in sorted(mc):
                keys.append(k)
                max_count.append(mc[k])
            key_off.append(len(keys))
            img_ref_off.append(len(tok_off) - 1)
        dev = self.dev
        i64 = lambda v: torch.tensor(v, dtype=torch.int64, device=dev)
        self._key_off, self._img_ref_off, self._tok_off = i64(key_off), i64(img_ref_off), i64(tok_off)
        self._keys = torch.from_numpy(np.array(keys or [0], dtype=np.uint64).view(np.int64)).to(dev)
        self._max_count = torch.tensor(max_count or [0], dtype=torch.int32, device=dev)
        self._toks = torch.tensor(toks or [0], dtype=torch.int32, device=dev)
        self._cider = CiderD.from_corpus(refs_per_image, device=dev, eos_id=self.eos, pad_id=self.pad)
        self.n_images = n
        self._stats = torch.zeros(n, 10, dtype=torch.int64, device=dev)     # BLEU: correct_1..4, guess_1..4, testlen, reflen
        self._rouge = torch.zeros(n, dtype=torch.float64, device=dev)
        self._cider_out = torch.zeros(n, dtype=torch.float64, device=dev)
        self._count = torch.zeros(n + 1, dtype=torch.int32, device=dev)     # hypotheses per image, then out-of-range indices
        self._out = torch.empty(9 + 6 * n, dtype=torch.float64, device=dev)

    def reset(self) -> None:
        """Forget the hypotheses added so far (the references stay)."""
        if self.n_images:
            self._count.zero_()

    def add(self, seq_words: torch.Tensor, image_idx) -> None:
        """seq_words int [H, L] word ids on the device; image_idx [H]: indices into the references given to ``set_refs``.
        Launches the three scoring kernels; no host synchronisation."""
        if not self.n_images:
            raise RuntimeError("call set_refs() with the split's reference captions first")
        if not seq_words.is_cuda:
            raise RuntimeError("CaptionMetrics.add runs on CUDA tensors only (there is no CPU fallback)")
        H, L = seq_words.shape
        if H == 0:
            return
        h = seq_words.to(torch.int32).contiguous()
        idx = torch.as_tensor(image_idx).to(self.dev, torch.int32).contiguous()
        if idx.shape != (H,):
            raise ValueError(f"image_idx has shape {tuple(idx.shape)}, expected ({H},)")
        n, s, c = self.n_images, lib.stream(), self._cider
        lib.call("sc_bleu_stats", lib.ptr(h), H, L, lib.ptr(idx), n, self.eos, self.pad, lib.ptr(self._key_off), lib.ptr(self._keys),
                 lib.ptr(self._max_count), lib.ptr(self._img_ref_off), lib.ptr(self._tok_off), lib.ptr(self._stats),
                 lib.ptr(self._count), lib.ptr(self._count[n:]), s)
        lib.call("sc_rouge_l", lib.ptr(h), H, L, lib.ptr(idx), n, self.eos, self.pad, lib.ptr(self._img_ref_off), lib.ptr(self._tok_off),
                 lib.ptr(self._toks), lib.ptr(self._rouge), s)
        r = c._refs
        lib.call("sc_cider_score", lib.ptr(h), H, L, lib.ptr(idx), n, self.eos, self.pad, lib.ptr(c.df_keys), lib.ptr(c.df_log), c.n_df,
                 c.ref_len, lib.ptr(r["img_off"]), lib.ptr(r["ng_off"]), lib.ptr(r["keys"]), lib.ptr(r["vec"]), lib.ptr(r["norm"]),
                 lib.ptr(self._cider_out), s)

    def compute(self) -> Tuple[Dict[str, float], torch.Tensor]:
        """One reduction launch and one device-to-host copy.  Raises ValueError unless every image of the split received exactly
        one hypothesis (coco-caption's ``assert gts.keys() == res.keys()``)."""
        if not self.n_images:
            raise RuntimeError("call set_refs() with the split's reference captions first")
        n = self.n_images
        lib.call("sc_caption_metrics_reduce", lib.ptr(self._stats), lib.ptr(self._rouge), lib.ptr(self._cider_out), lib.ptr(self._count),
                 lib.ptr(self._count[n:]), n, lib.ptr(self._out), lib.stream())
        out = self._out.cpu()
        missing, repeated, bad = (int(v) for v in out[6:9].tolist())
        if missing or repeated or bad:
            raise ValueError(f"every image needs exactly one hypothesis: {missing} of {n} images have none, {repeated} more than "
                             f"one, {bad} hypotheses have an image index outside [0, {n})")
        return dict(zip(METRICS, out[:6].tolist())), out[9:].view(n, 6)
