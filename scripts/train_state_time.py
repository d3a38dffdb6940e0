"""Cost of saving and restoring the trainer's optimizer state at the flagship size (bench.CFG = configs[1]: ORT 6x512, V = 10000,
~55 M weights and ~55 M mask logits), supermask, bf16, graph mode, seeded synthetic weights and a 50-image x 5-caption batch:
  export - OrtTrainer.optimizer_state_dict() (device-to-host copies of the four moment buffers, one CPU clone per parameter);
  save   - torch.save of that dict to a temporary file, and the file's size;
  load   - torch.load of the file, then OrtTrainer.load_optimizer_state_dict (host assembly, host-to-device copies).
Host wall-clock around work that ends in a device synchronise, median over --reps repetitions; a graphed train step is timed with
CUDA events beside them, so that a run can choose save_checkpoint_every.  The card's name and power limit are read in the same run.

    python scripts/train_state_time.py [--reps 5] [--out profiles/r07_train_state_time.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from sparse_caption_b200 import synthetic  # noqa: E402
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


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
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
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=0.0, device="cuda")
    tr = OrtTrainer(sd, cfg, mask_type="supermask", precision="bf16", seed=5, use_graph=True)

    def step():
        return tr.train_step(att, boxes, seqs, masks, seq_per_img=S, lr=1e-4, sparsity_target=0.9, sparsity_weight=5.0,
                             current_step=10, max_step=1000)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / a.steps
    export, save, load_file, load_state, size = [], [], [], [], None
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "optimizer_last.pth")
        for _ in range(a.reps + 1):    # (the first repetition warms the allocators and the page cache up: not counted)
            state, t_export = timed(tr.optimizer_state_dict)
            _, t_save = timed(lambda: torch.save(state, path))
            size = os.path.getsize(path)
            del state
            loaded, t_load_file = timed(lambda: torch.load(path))
            _, t_load = timed(lambda: tr.load_optimizer_state_dict(loaded))
            del loaded
            export.append(t_export)
            save.append(t_save)
            load_file.append(t_load_file)
            load_state.append(t_load)
    n_w = sum(tr.p[k].numel() for k in tr.names)
    n_s = sum(tr.s[k].numel() for k in tr.masked)
    med = lambda v: round(statistics.median(v[1:]), 1)   # noqa: E731
    row = {"config": "configs[1] (bench.CFG)", "mask_type": "supermask", "precision": "bf16", "graph": True, "weights": n_w,
           "mask_logits": n_s, "moment_bytes": 8 * (n_w + n_s), "export_ms": med(export), "torch_save_ms": med(save),
           "file_bytes": size, "torch_load_ms": med(load_file), "load_optimizer_state_dict_ms": med(load_state),
           "export_ms_all": [round(v, 1) for v in export[1:]], "load_ms_all": [round(v, 1) for v in load_state[1:]],
           "graphed_train_step_ms": round(step_ms, 2), "images": B, "captions_per_image": S, "reps": a.reps, "card": info}
    print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
