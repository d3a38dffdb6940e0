"""Time of one gradual-pruning mask update at the flagship size (bench.CFG = configs[1]: ORT 6x512, V = 10000, ~55 M masked
elements), bf16, graph mode, seeded synthetic weights and a 50-image x 5-caption batch, for mag_grad_uniform and mag_grad_blind:
  (a) trainer - OrtTrainer.update_masks_once on the trainer's own buffers (sc_prune_select, no host synchronisation);
  (b) host    - the path without it: model.sync_from_trainer() + model.update_masks_once (PruningMixin on the module) + the
                trainer rebuild that the changed parameters trigger + the first step after it (including its graph capture).
(a) is timed with CUDA events over --steps updates after --warmup; (b) wall-clock around work that ends in a device synchronise,
over --host-steps events.  A plain graphed train step is reported beside them.  The card's name and power limit are read in
the same run.

    python scripts/prune_update_time.py [--steps 20] [--warmup 3] [--host-steps 3] [--out profiles/r05_prune_update_time.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from sparse_caption_b200 import synthetic  # noqa: E402
from sparse_caption_b200 import relation_transformer as RT  # noqa: E402
from sparse_caption_b200.engine import ModelCfg  # noqa: E402
from sparse_caption_b200.trainer import OrtTrainer  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def batch(B, S, T, V):
    g = torch.Generator().manual_seed(4)
    seqs = torch.zeros(B * S, T + 1, dtype=torch.long)
    masks = torch.zeros(B * S, T + 1)
    for r in range(B * S):
        n = int(torch.randint(6, T - 1, (1,), generator=g))
        seqs[r, 0] = 2
        seqs[r, 1:1 + n] = torch.randint(4, V, (n,), generator=g)
        seqs[r, 1 + n] = 3
        masks[r, :n + 2] = 1
    return seqs, masks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    cfg = ModelCfg(bench.CFG)
    B, S, T = a.images, 5, cfg.max_seq_length
    att, boxes = synthetic.synthetic_inputs(B, bench.N_BOX, bench.CFG["att_feat_size"], seed=8888)
    att, boxes = att.cuda(), boxes.cuda()
    seqs, masks = batch(B, S, T, cfg.vocab_size)
    info = card()
    rows = []
    for mask_type in ("mag_grad_uniform", "mag_grad_blind"):
        sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=0.0, device="cuda")
        for k in [k for k, v in sd.items() if k.endswith(".weight") and v.dim() == 2]:
            sd[k + "_pruning_mask"] = torch.ones_like(sd[k])

        def step(tr):
            return tr.train_step(att, boxes, seqs, masks, seq_per_img=S, lr=1e-4)

        # (a) on the trainer's buffers
        tr = OrtTrainer(sd, cfg, mask_type=mask_type, precision="bf16", seed=5, use_graph=True)
        for _ in range(3):
            step(tr)
        targets = [0.5 + 0.02 * (i % 10) for i in range(a.warmup + a.steps)]
        for s in targets[: a.warmup]:
            tr.update_masks_once(s)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in targets[a.warmup:]:
            tr.update_masks_once(s)
        e1.record()
        torch.cuda.synchronize()
        trainer_ms = e0.elapsed_time(e1) / a.steps
        masked = sum(tr.s[k].numel() for k in tr.active_masked())
        e0.record()
        for _ in range(a.steps):
            step(tr)
        e1.record()
        torch.cuda.synchronize()
        step_ms = e0.elapsed_time(e1) / a.steps
        del tr
        torch.cuda.empty_cache()

        # (b) the module path: sync, PruningMixin on the module, rebuild, first step (capture included)
        model = RT.get_model("relation_transformer_prune")(dict(bench.CFG, prune_type=mask_type)).cuda()
        model.load_state_dict(sd, strict=False)
        model.precision = "bf16"
        tr = model.trainer(seed=5, use_graph=True)
        for _ in range(3):
            step(tr)
        host = []
        for i in range(a.host_steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.sync_from_trainer()
            model.update_masks_once(0.5 + 0.02 * i)
            tr = model.trainer(seed=5, use_graph=True)
            step(tr)
            torch.cuda.synchronize()
            host.append((time.perf_counter() - t0) * 1e3)
        del model, tr
        torch.cuda.empty_cache()
        row = {"mask_type": mask_type, "masked_elements": masked, "precision": "bf16", "graph": True, "images": B,
               "captions_per_image": S, "trainer_update_ms": round(trainer_ms, 3), "host_path_ms": [round(v, 1) for v in host],
               "host_over_trainer": round(min(host) / trainer_ms, 1), "graphed_train_step_ms": round(step_ms, 2),
               "steps": a.steps, "warmup": a.warmup, "card": info}
        rows.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
