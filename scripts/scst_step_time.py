"""SCST training step time at the flagship size (bench.CFG = configs[1]/[4]: ORT 6x512, V = 10000, 50 images x 36 boxes, L = 16),
seeded synthetic weights and inputs, bf16:
  (a) module  - the module-tree recipe (ModuleTrainer.scst_step: train-mode engine rebuilt for every rollout, eval-mode engine for
                the greedy baseline, autograd re-score, one clip + Adam launch per tensor);
  (b) eager   - OrtTrainer.scst_step with use_graph=False (bound rollout engine, fused teacher-forcing step, eager launches);
  (c) graphed - OrtTrainer.scst_step with use_graph=True (the engine's graphs + one trainer graph).
Masks: fixed 0/1 masks at bench.SPARSITY (mask_freeze) and supermask logits.  Rollouts: beam 5 + greedy baseline, and 5
multinomial samples with the mean-of-others baseline.  CUDA events around the timed steps after warm-up; one JSON line per
setting with the card's name and power limit read in the same run.

    python scripts/scst_step_time.py [--steps 10] [--warmup 3] [--out profiles/r04_scst_step_time.json]
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
from sparse_caption_b200 import relation_transformer as RT  # noqa: E402
from sparse_caption_b200.cider import CiderD  # noqa: E402
from sparse_caption_b200.engine import ModelCfg  # noqa: E402
from sparse_caption_b200.trainer import ModuleTrainer, OrtTrainer  # noqa: E402

ROLLOUTS = [("beam5_greedy", {"beam_size": 5}, "greedy"),
            ("sample5_mean", {"num_random_sample": 5, "beam_size": 0}, "sample")]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def state_dict(cfg, mask_type):
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=0.0, device="cuda")
    g = torch.Generator(device="cpu").manual_seed(7)
    for k in [k for k, v in sd.items() if k.endswith(".weight") and v.dim() == 2]:
        keep = (torch.rand(sd[k].shape, generator=g) >= bench.SPARSITY).float().cuda()
        sd[k + "_pruning_mask"] = keep if mask_type == "mask_freeze" else keep * 6.0 - 3.0   # supermask: logits +-3
    return sd


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--module-steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    cfg = ModelCfg(bench.CFG)
    B = a.images
    att, boxes = synthetic.synthetic_inputs(B, bench.N_BOX, bench.CFG["att_feat_size"], seed=8888)
    att, boxes = att.cuda(), boxes.cuda()
    # references: five random 9-word captions per image over the first 500 ids (random weights sample across the vocabulary, so
    # most rewards are small; the step's work does not depend on their values)
    g = torch.Generator().manual_seed(3)
    refs = [[torch.randint(4, 500, (9,), generator=g).tolist() for _ in range(5)] for _ in range(B)]
    scorer = CiderD.from_corpus(refs, device="cuda")
    info = card()
    rows = []
    for mask_type in ("mask_freeze", "supermask"):
        sd = state_dict(cfg, mask_type)
        for name, opt, baseline in ROLLOUTS:
            kw = dict(scorer=scorer, opt=opt, baseline=baseline, lr=1e-5, mask_lr=1e-3)
            res = {}
            model = RT.get_model("relation_transformer_prune")(dict(bench.CFG, prune_type=mask_type)).cuda()
            model.load_state_dict({k: v for k, v in sd.items()}, strict=False)
            model.precision = "bf16"
            mt = ModuleTrainer(model)
            res["module_ms"] = timed(lambda: mt.scst_step(att, boxes, **kw), a.module_steps, 1)
            del model, mt
            for graph in (False, True):
                tr = OrtTrainer(sd, cfg, mask_type=mask_type, precision="bf16", seed=5, use_graph=graph)
                res["graphed_ms" if graph else "eager_ms"] = timed(lambda: tr.scst_step(att, boxes, **kw), a.steps, a.warmup)
                del tr
            torch.cuda.empty_cache()
            row = {"masks": mask_type, "rollout": name, "opt": opt, "baseline": baseline, "images": B,
                   "captions_per_image": 5, "L": cfg.max_seq_length, "precision": "bf16"}
            row.update({k: round(v, 2) for k, v in res.items()})
            row["module_over_graphed"] = round(res["module_ms"] / res["graphed_ms"], 2)
            row.update({"steps": a.steps, "module_steps": a.module_steps, "warmup": a.warmup, "card": info})
            rows.append(row)
            print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
