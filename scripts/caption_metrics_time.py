"""Time of the validation scores of one split: 5000 images x 5 references (lengths 6-16), seeded synthetic word ids (a
Zipf-like vocabulary of 10000 words; each hypothesis shares a random stretch with one of its references, so n-grams match).
  (a) device - CaptionMetrics.add over batches of --batch hypotheses + compute() (three scoring launches per batch, one reduction,
               one device-to-host copy), CUDA events over --steps passes after --warmup; set_refs (once per split) separately;
  (b) host   - the oracle (oracle/caption_metrics_oracle.py, a literal Python restatement of bleu_scorer.py / rouge.py /
               cider_scorer.py on word ids) on the same captions, wall clock, once.  It is not coco-caption itself: the PTB
               tokenizer's Java round trip and the detokenisation of the captions are not in it.
Whether (a) and (b) agree is recorded.  The card's name and power limit are read in the same run.

    python scripts/caption_metrics_time.py [--out profiles/r06_caption_metrics_time.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import caption_metrics_oracle as M  # noqa: E402
from sparse_caption_b200.metrics import CaptionMetrics  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def split(n_img, n_ref, L, seed=0, vocab=10000):
    rng = np.random.RandomState(seed)
    p = 1.0 / np.arange(1, vocab + 1)
    p /= p.sum()
    draw = lambda n: [int(w) + 4 for w in rng.choice(vocab, n, p=p)]
    refs = [[draw(rng.randint(6, 17)) for _ in range(n_ref)] for _ in range(n_img)]
    hyps, rows = [], np.zeros((n_img, L), dtype=np.int32)
    for i in range(n_img):
        n = rng.randint(6, 17)
        src = refs[i][rng.randint(n_ref)]
        a = rng.randint(len(src))
        h = (draw(rng.randint(0, 4)) + src[a: a + rng.randint(2, 9)] + draw(n))[:n]
        hyps.append(h)
        rows[i, :n] = h
        if n < L:
            rows[i, n] = 3
    return refs, hyps, torch.from_numpy(rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--refs", type=int, default=5)
    ap.add_argument("--batch", type=int, default=500)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    L = 20
    refs, hyps, rows = split(a.images, a.refs, L)
    m = CaptionMetrics(device="cuda")
    t0 = time.perf_counter()
    m.set_refs(refs)
    torch.cuda.synchronize()
    t_refs = time.perf_counter() - t0
    seq = rows.cuda()
    idx = torch.arange(a.images, device="cuda")
    chunks = [(seq[i: i + a.batch], idx[i: i + a.batch]) for i in range(0, a.images, a.batch)]

    def one_pass():
        m.reset()
        for s, j in chunks:
            m.add(s, j)
        return m.compute()

    for _ in range(a.warmup):
        one_pass()
    times = []
    for _ in range(a.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        scores, per = one_pass()          # compute() ends in the device-to-host copy
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    t0 = time.perf_counter()
    want, want_per = M.evaluate(hyps, refs)
    t_host = time.perf_counter() - t0
    rel = max(abs(scores[k] - want[k]) / max(abs(want[k]), 1e-300) for k in M.METRICS)
    per_err = float(np.max(np.abs(per.numpy() - want_per) / np.maximum(np.abs(want_per), 1e-15)))
    res = {
        "card": card(), "images": a.images, "refs_per_image": a.refs, "ref_len": "6-16", "hyp_len": "6-16", "batch": a.batch,
        "device_add_compute_ms": {"median": float(np.median(times)), "min": float(np.min(times)), "max": float(np.max(times)),
                                  "passes": a.steps, "warmup": a.warmup},
        "set_refs_host_s": t_refs, "oracle_host_s": t_host,
        "scores_device": scores, "scores_oracle": want,
        "max_rel_diff_corpus": rel, "max_rel_diff_per_image": per_err, "agree_1e-12": bool(rel <= 1e-12 and per_err <= 1e-12),
    }
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
