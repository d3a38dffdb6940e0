"""Diverse beam search (group_size > 1) decode time on the flagship configuration (bench.CFG, bench.SPARSITY, configs[2]):
512 images already on the device, the encoder run once, then each decode setting's CUDA graph replayed after warm-up and
timed with CUDA events.  Prints one JSON line per setting (ms per 512-image decode, captions/s counted as images/s like
bench.py, kernel launches per decode) and the card's name and power limit read in the same run.

    python scripts/diverse_beam_time.py [--reps 30] [--out profiles/r03_diverse_beam_time.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from sparse_caption_b200 import synthetic  # noqa: E402
from sparse_caption_b200.engine import ModelCfg, OrtEngine  # noqa: E402

SETTINGS = [("beam3_g1", {"beam_size": 3}, True),
            ("beam3_g3_l0.5", {"beam_size": 3, "group_size": 3, "diversity_lambda": 0.5}, True),
            ("beam6_g2_l0.5", {"beam_size": 6, "group_size": 2, "diversity_lambda": 0.5}, True),
            ("beam3_g3_l0.5_nofuse", {"beam_size": 3, "group_size": 3, "diversity_lambda": 0.5}, False)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    cfg = ModelCfg(bench.CFG)
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=bench.SPARSITY, device="cuda")
    att, boxes = synthetic.synthetic_inputs(a.images, 36, bench.CFG["att_feat_size"], seed=8888)
    att, boxes = att.cuda(), boxes.cuda()
    engines = {True: OrtEngine(sd, cfg, precision="bf16"), False: OrtEngine(sd, cfg, precision="bf16", fuse_topk=False)}
    encs = {k: e.encode(att, boxes) for k, e in engines.items()}
    rows = []
    info = card()
    for name, opt, fused in SETTINGS:
        eng, enc = engines[fused], encs[fused]
        for _ in range(a.warmup):
            eng.decode(enc, opt)
        ws = next(w for w in eng._dec_ws.values() if getattr(w, "opt_key", None) is not None and w.opt_key[1:] ==
                  (tuple(sorted((k, str(v)) for k, v in opt.items())),))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            eng.decode(enc, opt)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.reps
        b = int(opt["beam_size"])
        g = int(opt.get("group_size", 1))
        row = {"setting": name, "opt": opt, "fuse_topk": fused, "images": a.images,
               "captions_per_image": (b // g) * g, "ms_per_decode": round(ms, 3),
               "captions_per_s": round(a.images / ms * 1e3, 1), "launches_per_decode": ws.launches,
               "reps": a.reps, "card": info}
        rows.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
