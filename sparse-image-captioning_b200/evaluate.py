"""The caller after the path (SURVEY.md section 8f.1): ``TrainingModule.eval_on_split`` (utils/training.py:257-327) up to the
caption JSON - batches -> ``mode="sample"`` -> token ids on the host -> detokenisation -> COCO-caption result file
(data/karpathy.py:193-221), and optionally coco-caption's BLEU-1..4 / ROUGE-L / CIDEr on the device (``metrics.CaptionMetrics``,
fed the best captions as word ids before they leave the GPU).  METEOR / SPICE / PTBTokenizer (Java) are out of scope.

Detokenisation: word-level tokenizers call ``tokenizer.decode`` per caption (SentencePiece, C++); radix tokenizers (ACORT) first
map the radix digits to word ids for the WHOLE batch in one vectorised pass on the device (detok.radix_to_word_ids), so the
Python loop only sees word ids.
"""
import json
import os
import time
from typing import Callable, Iterable, List, Optional, Sequence, Tuple

import torch

from .detok import radix_to_word_ids


def best_captions(seq: torch.Tensor) -> torch.Tensor:
    """[B, beam, L] -> [B, L]: ``seq[k][0]``, the highest-scoring beam (training.py:273)."""
    return seq[:, 0]


def detokenize(seq: torch.Tensor, *, decode_words: Callable[[List[int]], str], radix: Optional[Tuple[int, int]] = None, eos_id: int = 3,
               pad_id: int = 0, vocab_len: Optional[int] = None) -> List[str]:
    """Token ids [B, L] -> caption strings.  ``radix=(radix_base, tokens_per_word)``: ACORT's radix re-encoding
    (tokenizer.py:583-647); word ids beyond the word vocabulary map to <unk> = 1 as in the reference (:640)."""
    if radix is not None:
        base, tpw = radix
        words, n = radix_to_word_ids(seq, base, tpw)
        words, n = words.cpu(), n.cpu()
        out = []
        for i in range(words.shape[0]):
            ids = words[i, : int(n[i])].tolist()
            if vocab_len is not None:
                ids = [w if w < vocab_len else 1 for w in ids]
            sent = decode_words(ids).replace("<unk>", " <unk>")
            out.append(sent[1:] if sent.startswith(" ") else sent)
        return out
    s = seq.cpu().tolist()
    out = []
    for ids in s:
        if eos_id in ids:
            ids = ids[: ids.index(eos_id)]
        out.append(decode_words([t for t in ids if t != pad_id]))
    return out


def coco_caption_json_dump(image_ids_and_captions: Iterable[Tuple[int, str]], output_fpath: str) -> str:
    """data/karpathy.py:193-221: ``[{"image_id": id, "caption": str}, ...]`` (image ids already resolved by the dataset)."""
    assert output_fpath.endswith(".json"), f"`output_fpath` should end with `.json`, saw `{output_fpath}` instead."
    coco_json = []
    for image_id, caption in image_ids_and_captions:
        assert isinstance(caption, str), "Caption must be a string."
        coco_json.append({"image_id": image_id, "caption": caption})
    os.makedirs(os.path.split(output_fpath)[0] or ".", exist_ok=True)
    with open(output_fpath, "w") as f:
        json.dump(coco_json, f)
    return output_fpath


def eval_on_split(engine_or_model, batches: Iterable[dict], opt: dict, *, decode_words: Callable[[List[int]], str],
                  radix: Optional[Tuple[int, int]] = None, vocab_len: Optional[int] = None, json_fpath: Optional[str] = None,
                  eos_id: int = 3, metrics=None):
    """``batches`` yield {"att_feats", "boxes", "att_masks" (optional), "image_ids"}.  Returns (predictions, images / s, json path).

    ``metrics``: a ``CaptionMetrics`` whose ``set_refs`` holds the split's references; every batch then also yields "image_idx",
    the images' indices into those references (not the COCO image ids of the JSON), and its best captions are added to it as word
    ids on the device (radix models: ``radix_to_word_ids``, ids beyond ``vocab_len`` -> <unk> as in ``detokenize``).  The
    caller reads ``metrics.compute()``."""
    t0 = time.perf_counter()
    ids, preds = [], []
    for data in batches:
        if hasattr(engine_or_model, "sample"):
            seq, _ = engine_or_model.sample(data["att_feats"], data["boxes"], data.get("att_masks"), opt)
        else:
            seq, _ = engine_or_model(att_feats=data["att_feats"], boxes=data["boxes"], att_masks=data.get("att_masks"), opt=opt, mode="sample")
        best = best_captions(seq)
        if metrics is not None:
            words = best
            if radix is not None:
                words, _ = radix_to_word_ids(best, *radix)
                if vocab_len is not None:
                    words = torch.where(words < vocab_len, words, torch.ones_like(words))
            metrics.add(words, data["image_idx"])
        preds += detokenize(best, decode_words=decode_words, radix=radix, vocab_len=vocab_len, eos_id=eos_id)
        ids += list(data["image_ids"])
    speed = len(ids) / max(time.perf_counter() - t0, 1e-9)
    path = coco_caption_json_dump(zip(ids, preds), json_fpath) if json_fpath else None
    return preds, speed, path
