"""Beam search decode time at 3 to 32 beams on the flagship configuration (bench.CFG, bench.SPARSITY, configs[2]): 512 images
already on the device, the encoder run once, then each beam width's CUDA graph replayed after warm-up and timed with CUDA
events on one stream.  Beams 3, 5 and 8 run the per-thread-list beam step (3 and 5 on the fused generator + top-k records),
10, 16 and 32 the radix-select row pass and merge on materialised logits.

A separate torch.profiler run (eager launches, the same kernels) gives the row-pass, merge and cross-attention kernel times
at beams 8, 10 and 32; the row pass is also given as GB/s of logits read, next to the bandwidth of a 2 GB device-to-device
copy (bytes read + written) measured in the same run.  The card's name, power limit and max SM clock are read in the same run.

    python scripts/wide_beam_time.py [--reps 30] [--out profiles/r08_wide_beam_time.json]
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

BEAMS = [3, 5, 8, 10, 16, 32]
PROFILED = [8, 10, 32]
KERNELS = {"row_pass": ("beam_row_kernel", "beam_row_wide_kernel", "beam_row_partials_kernel"),
           "merge": ("beam_merge_kernel", "beam_merge_wide_kernel"),
           "cross_attn": ("cross_attn_mma_kernel", "cross_attn_mma_wide_kernel", "cross_attn_step_kernel",
                          "cross_attn_step_wide_kernel")}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def copy_gbps(nbytes=2 << 30, reps=20):
    src = torch.empty(nbytes // 4, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def kernel_kind(name):
    """(kind, kernel name) of a profiled kernel, (None, None) when it is not one of KERNELS."""
    for kind, names in KERNELS.items():
        for n in names:
            if f"::{n}<" in name or f"::{n}(" in name:
                return kind, n
    return None, None


def profile_kernels(eng, enc, opt, reps):
    from torch.profiler import ProfilerActivity, profile
    eng.decode(enc, opt)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            eng.decode(enc, opt)
        torch.cuda.synchronize()
    out = {k: {"us_per_decode": 0.0, "launches_per_decode": 0, "names": []} for k in KERNELS}
    for ev in prof.key_averages():
        kind, kname = kernel_kind(ev.key)
        if kind is None:
            continue
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        out[kind]["us_per_decode"] += t / reps
        out[kind]["launches_per_decode"] += ev.count // reps
        if kname not in out[kind]["names"]:
            out[kind]["names"].append(kname)
    for v in out.values():
        v["us_per_decode"] = round(v["us_per_decode"], 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    cfg = ModelCfg(bench.CFG)
    L, V = cfg.max_seq_length, cfg.vocab_size
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=bench.SPARSITY, device="cuda")
    att, boxes = synthetic.synthetic_inputs(a.images, 36, bench.CFG["att_feat_size"], seed=8888)
    att, boxes = att.cuda(), boxes.cuda()
    info = card()
    eng = OrtEngine(sd, cfg, precision="bf16")
    enc = eng.encode(att, boxes)
    result = {"card": info, "config": "configs[2] (bench.CFG, bf16, synthetic weights and inputs)", "images": a.images,
              "decode": [], "kernels": {}}
    for beam in BEAMS:
        opt = {"beam_size": beam}
        for _ in range(a.warmup):
            eng.decode(enc, opt)
        ws = eng._get_dec_ws(enc.B, beam, enc.N, False, enc.slot)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            eng.decode(enc, opt)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.reps
        row = {"beam": beam, "ms_per_decode": round(ms, 3), "captions_per_s": round(a.images / ms * 1e3, 1),
               "launches_per_decode": ws.launches, "fused_topk": ws.topk_part is not None, "reps": a.reps}
        result["decode"].append(row)
        print(json.dumps(row), flush=True)
    del eng, enc
    torch.cuda.empty_cache()
    result["copy_GBps"] = round(copy_gbps(), 1)
    eager = OrtEngine(sd, cfg, precision="bf16", use_graphs=False)
    enc = eager.encode(att, boxes)
    for beam in PROFILED:
        k = profile_kernels(eager, enc, {"beam_size": beam}, a.profile_reps)
        rows_read = a.images * (1 + (L - 1) * beam)  # t = 0 expands one row per image
        if k["row_pass"]["us_per_decode"] > 0 and beam > 5:  # (beams <= 5 read top-k records, not logits)
            k["row_pass"]["logits_GBps"] = round(rows_read * V * 4 / (k["row_pass"]["us_per_decode"] * 1e-6) / 1e9, 1)
        result["kernels"][str(beam)] = k
        print(json.dumps({"beam": beam, **k}), flush=True)
    print(json.dumps({"copy_GBps": result["copy_GBps"], "card": info}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
