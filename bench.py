"""Benchmark of the B200-native ORT / ACORT captioning hot path: one JSON result line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config infer|train|acort|scst] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`; synthetic 36-region x 2048-d features + boxes, random-init randomly pruned weights):
  infer (default, configs[2]): ORT 6x512, 95 % sparse binarized-mask weights, beam-3 incremental decoding, L = 16, 512 images
                               per GPU per step; the line also carries the SMP training arm (configs[1]) under "train".
  train (configs[1]):          ORT supermask (SMP) training, bf16 GEMMs / fp32 master weights + logits, 50 images x 5 captions per
                               GPU per step, Bernoulli masks + dropout + sparsity loss + clip + Adam; NCCL all-reduce of dWm at N > 1.
  acort (configs[3]):          ACORT (2 unique layers x 3, share_att 'kv'), radix vocabulary 771, 99.1 % sparse, beam 5, L = 26.
  scst  (configs[4]):          SCST rollouts for ORT: beam-5 + greedy baseline decode over ONE encoder pass, 1024 images per step.
A "step" = one batch through encoder + all decode steps + beam bookkeeping (train: one full optimizer step).
N > 1: one process per GPU (torchrun), images sharded by rank, no collective on the inference data path (weak scaling).

  value : metric with inputs already resident in HBM.
  e2e   : same through OrtEngine.submit() with pinned HOST fp32 features / boxes (H2D inside the timed region) and a
          device->host read of the decoded tokens + log-probs every step.  "e2e_bf16_host": same with bf16 pinned features.
  roofline     : dominant kernel family (the tcgen05 GEMM): algorithmic FLOPs / in-graph CUDA-event time of every GEMM launch
                 of one step, alone and with the timed region's concurrency, against MEASURED_PEAKS.json; "hbm_kernels": the
                 HBM-bound decode kernels (cross / self attention, LayerNorm) as GB/s against the measured copy bandwidth.
  cpu_baseline : the CPU oracle (a port of the reference's PyTorch path) on this box's host cores, bounded sample.
  --dump-outputs DIR : after the timed steps, what the timed path returned for its last step as DIR/<name>.npy (float32 /
                 float64, rank 0): infer / acort / scst the tokens (beam<b>_seq) and log-probs (beam<b>_logprobs) of each decode
                 of the last timed device launch, [images, b, L]; train the loss and a seeded sample of the weights and mask
                 logits the last step left.  Inputs are seeded, so two builds run with the same arguments can be compared file
                 by file.
  --impl reference : the same CPU arm alone (the reference is pure Python/PyTorch; its hot path restated in
                 oracle/ort_oracle.py is what runs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG = dict(d_model=512, dim_feedforward=2048, num_layers=6, num_heads=8, max_seq_length=16, att_feat_size=2048,
           vocab_size=10000)
ACORT_CFG = dict(CFG, vocab_size=771, max_seq_length=26, share_att_encoder="kv", share_att_decoder="kv",
                 share_layer_encoder=(0, 0, 0, 1, 1, 1), share_layer_decoder=(0, 0, 0, 1, 1, 1), bos_token_id=769, eos_token_id=770)
SPARSITY = 0.95
BEAM = 3
N_BOX = 36
WORKLOADS = {
    "infer": dict(cfg=CFG, sparsity=0.95, decodes=[{"beam_size": 3}], images=512, metric="ort95_beam3_captions_per_sec", unit="captions/s",
                  label="ORT 6x512 95%-sparse binarized-mask beam-3 inference, L=16, V=10000, 36x2048 features + boxes", idx=2),
    "acort": dict(cfg=ACORT_CFG, sparsity=0.991, decodes=[{"beam_size": 5}], images=512, metric="acort991_beam5_captions_per_sec",
                  unit="captions/s", label="ACORT (2 unique layers x 3, share_att kv) 99.1%-sparse radix-vocabulary (771) beam-5 "
                  "incremental decoding, L=26, 36x2048 features + boxes", idx=3),
    "scst": dict(cfg=CFG, sparsity=0.95, decodes=[{"beam_size": 5}, {"beam_size": 1}], images=1024, metric="scst_rollout_images_per_sec",
                 unit="images/s", label="SCST rollout for ORT (fixed 0/1 masks): beam-5 rollout + greedy baseline decode over one encoder "
                 "pass, L=16, V=10000 (CIDEr scoring excluded)", idx=4),
}
METRIC = WORKLOADS["infer"]["metric"]
UNIT = WORKLOADS["infer"]["unit"]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each decode GEMM shape, from the committed ncu capture
    (scripts/ncu_gemm_traffic.sh -> profiles/r02_gemm_traffic.json, keys "M,N,K,out_bytes,residual")."""
    p = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def write_outputs(path, arrays, cap=64 << 20):
    """--dump-outputs: each array as <path>/<name>.npy, float64 kept, everything else as float32 (token ids are exact there).
    Above `cap` bytes in all, the arrays (which then must share their leading, per-image dimension) keep the same fixed,
    seeded sample of rows, in order, and rows.npy lists the kept indices."""
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > cap:
        lead = {v.shape[0] for v in arrays.values()}
        assert len(lead) == 1, f"cannot sample arrays of different leading dimensions {sorted(lead)} down to {cap} bytes"
        n = lead.pop()
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * cap // (total + 8 * n)), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays["rows"] = keep.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arms (reference arm / cpu_baseline): the oracle port of the reference's PyTorch path on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def cpu_arm(steps, warmup, images, wl=None):
    from oracle import ort_oracle as O
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200 import synthetic
    wl = wl or WORKLOADS["infer"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = ModelCfg(wl["cfg"])
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=wl["sparsity"])
    ocfg = O.Cfg(**wl["cfg"])
    att, boxes = synthetic.synthetic_inputs(images, N_BOX, wl["cfg"]["att_feat_size"], seed=8888)

    def one(a, b):
        memory, src_mask = O.encode(sd, ocfg, a, b, None)  # encoder once, every decode of the step shares it
        for opt in wl["decodes"]:
            if opt.get("beam_size", 1) > 1:
                O.beam_search(sd, ocfg, memory, src_mask, opt)
            else:
                O.greedy_search(sd, ocfg, memory, src_mask, opt)

    with torch.no_grad():
        for _ in range(warmup):
            one(att[:8], boxes[:8])
        t0 = time.perf_counter()
        for _ in range(steps):
            one(att, boxes)
        dt = time.perf_counter() - t0
    return images * steps / dt, dt / steps, cores


def _train_batch(B, S, T, V, rank):
    from sparse_caption_b200 import synthetic
    g = torch.Generator().manual_seed(8888 + rank)
    att, boxes = synthetic.synthetic_inputs(B, N_BOX, CFG["att_feat_size"], seed=8888 + rank, pin=torch.cuda.is_available())
    R = B * S
    seqs = torch.zeros(R, T + 1, dtype=torch.long)
    masks = torch.zeros(R, T + 1)
    lens = torch.randint(6, T - 1, (R,), generator=g)
    for r in range(R):
        n = int(lens[r])
        seqs[r, 0] = 2
        seqs[r, 1:1 + n] = torch.randint(4, V, (n,), generator=g)
        seqs[r, 1 + n] = 3
        masks[r, :n + 2] = 1
    return att, boxes, seqs, masks


def cpu_train_arm(steps, warmup, images):
    """SMP training step of the reference path on the host cores: supermask forward (sigmoid -> Bernoulli -> mul per masked
    layer, masked_layer.py:84-110) + LanguageModelCriterion + backward through the straight-through estimators, fp32 autograd
    over the oracle, clip + the two Adam groups over 110 M parameters included."""
    from oracle import ort_oracle as O
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200 import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg_d = dict(CFG, max_seq_length=17)
    ocfg = O.Cfg(**cfg_d)
    sd = synthetic.random_state_dict(ModelCfg(cfg_d), seed=1234, sparsity=0.0)
    W = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point()}
    keys = [k for k in sd if k.endswith(".weight") and sd[k].dim() == 2]
    Sg = {k: torch.full_like(sd[k], 5.0).requires_grad_(True) for k in keys}
    opt = torch.optim.Adam([{"params": list(W.values()), "lr": 3e-4, "betas": (0.9, 0.98), "eps": 1e-9},
                            {"params": list(Sg.values()), "lr": 100.0, "betas": (0.9, 0.98), "eps": 1e-2}])
    att, boxes, seqs, masks = _train_batch(images, 5, 17, CFG["vocab_size"], 0)

    def step():
        opt.zero_grad()
        eff = dict(W)
        for k in keys:
            p = torch.sigmoid(Sg[k])
            m = torch.bernoulli(p.detach())
            eff[k] = (p + (m - p).detach()) * W[k]
        lp = O.forward_tf(eff, ocfg, att, boxes, seqs, None)
        loss = O.lm_criterion(lp, seqs[:, 1:], masks[:, 1:])
        loss.backward()
        for g in opt.param_groups:
            torch.nn.utils.clip_grad_value_(g["params"], 0.1)
        opt.step()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return images * steps / dt, dt / steps, cores


# ----------------------------------------------------------------------------------------------------------------------
# in-graph kernel timing helpers (roofline legs)
# ----------------------------------------------------------------------------------------------------------------------
def _time_graph(run, dev, reps=40):
    """us per launch of run(i): `reps` launches captured in one CUDA graph on the current stream, CUDA events around two replays."""
    run(0)
    torch.cuda.synchronize(dev)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for i in range(reps):
            run(i)
    gr.replay()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); gr.replay(); gr.replay(); e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) * 1e3 / (2 * reps)


def time_train_gemms(prof, dev):
    """Every distinct GEMM launch of one training step (forward with its dropout / residual epilogue, dX, dX with the
    activation-mask epilogue, weight gradient incl. its split-K reduction) re-issued through the same entry point, 20 launches
    inside one CUDA graph, CUDA events around two replays: microseconds without the host's launch gaps.  Returns
    (total us per step, total flop per step)."""
    from sparse_caption_b200 import kernels as KK
    groups = {}
    for name, meta, a, b in prof:
        if meta and meta[0] == "gemm_bf16":
            key = (name,) + tuple(meta[1:])
            groups[key] = groups.get(key, 0) + 1
    tot_us, tot_fl = 0.0, 0.0
    for key, cnt in groups.items():
        name, d1, d2, d3 = key[:4]
        if name == "sc_linear_wgrad_rowmajor":
            N, Kd, M = d1, d2, d3
            dy = torch.randn(M, N, device=dev).bfloat16(); x = torch.randn(M, Kd, device=dev).bfloat16()
            W = torch.randn(N, Kd, device=dev)
            gW = torch.empty_like(W)
            wsb = torch.empty(4 * N * Kd, device=dev)
            run = lambda i: KK.linear_wgrad_rowmajor(dy, x, W, None, KK.MASK_NONE, gW, None, workspace=wsb)
            fl = 2.0 * M * N * Kd
        else:
            M, N, Kd = d1, d2, d3
            ys = key[6]
            x = torch.randn(M, Kd, device=dev).bfloat16(); w = torch.randn(N, Kd, device=dev).bfloat16()
            outs = [torch.empty(M, N, device=dev, dtype=torch.bfloat16 if ys == 2 else torch.float32) for _ in range(2)]
            fl = 2.0 * M * N * Kd
            if name == "sc_linear_hmask":
                h = torch.randn(M, N, device=dev).clamp_min(0).bfloat16(); cs = torch.zeros(N, device=dev)
                run = lambda i: KK.linear_hmask(x, w, h, outs[i % 2], scale=1.1, colsum=cs)
            elif name == "sc_linear_dropout":
                has_res, relu, drop, tile = key[8], key[9], key[10], key[11]
                bias = torch.randn(N, device=dev); res = torch.randn(M, N, device=dev) if has_res else None
                run = lambda i: KK.linear_dropout(x, w, bias, residual=res, relu=relu, out=outs[i % 2], p=0.1 if drop else 0.0,
                                                  drop_seed=1, drop_stream=2, tile_n=tile)
            else:
                has_res = key[8] if len(key) > 8 else False
                res = torch.randn(M, N, device=dev) if has_res else None
                run = lambda i: KK.linear(x, w, None, residual=res, out=outs[i % 2])
        us = _time_graph(run, dev, 20)
        if os.environ.get("SC_BENCH_VERBOSE") == "1":
            print(f"  train gemm {name:26s} {str(key[1:4]):22s} x{cnt:3d}  {us:7.2f} us  {fl / us / 1e6:6.0f} TF/s  flags {key[4:]}", file=sys.stderr)
        tot_us += us * cnt
        tot_fl += fl * cnt
    return tot_us, tot_fl


def hbm_kernel_roofline(dev, B, beam, N, cfg, peaks):
    """The HBM-bound decode kernels (K5 self attention at mid / last step, K6 cross attention, K9 LayerNorm) timed alone in a
    CUDA graph over 4 rotating buffer sets (together larger than the 126 MB L2), algorithmic bytes / time against the measured
    copy bandwidth."""
    from sparse_caption_b200 import kernels as KK
    d, h, L = cfg["d_model"], cfg["num_heads"], cfg["max_seq_length"]
    R = B * beam
    bf = dict(device=dev, dtype=torch.bfloat16)
    out = []

    def entry(name, run, nbytes):
        us = _time_graph(run, dev)
        gbs = nbytes / us / 1e3
        out.append({"kernel": name, "us_per_launch": us, "algorithmic_bytes": nbytes, "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": gbs / peaks["hbm"]})

    C = 4
    qc = [torch.randn(R, d, **bf) for _ in range(C)]
    mkv = [torch.randn(B * N, 2 * d, **bf) for _ in range(C)]
    att = torch.empty(R, d, **bf)
    entry("sc_decode_cross_attn_step", lambda i: KK.cross_attn_step(qc[i % C], mkv[i % C][:, 0:], mkv[i % C][:, d:], None, att, B=B, beam=beam,
                                                                    N=N, D=d, h=h, ldq=d, ldm=2 * d, ldo=d),
          B * N * 2 * d * 2 + 2 * R * d * 2)
    qkv = [torch.randn(R, 3 * d, **bf) for _ in range(C)]
    ck = [torch.randn(L, R, d, **bf) for _ in range(C)]
    cv = [torch.randn(L, R, d, **bf) for _ in range(C)]
    anc = torch.arange(R, device=dev, dtype=torch.int32).unsqueeze(1).expand(R, L).contiguous()
    for t in (L // 2, L - 1):
        entry(f"sc_decode_self_attn_step(t={t})",
              lambda i, t=t: KK.self_attn_step(qkv[i % C][:, 0:], qkv[i % C][:, d:], qkv[i % C][:, 2 * d:], ck[i % C], cv[i % C], anc, att, R=R, D=d,
                                               h=h, n_prev=t, write_slot=t, ldq=3 * d, ldk=3 * d, ldv=3 * d, ldo=d, anc_ld=L, slot_div=1),
              R * (t + 1) * 2 * d * 2 + R * 3 * d * 2 + 2 * R * d * 2 + R * d * 2)
    rows = B * N  # the encoder-sized LayerNorm (the decode-sized one, R rows, moves 4.7 MB and is launch-latency bound)
    x = [torch.randn(rows, d, device=dev) for _ in range(C)]
    xn = torch.empty(rows, d, **bf)
    a2, b2 = torch.ones(d, device=dev), torch.zeros(d, device=dev)
    entry(f"sc_layernorm({rows} rows)", lambda i: KK.layernorm(x[i % C], a2, b2, out=xn), rows * d * 6)
    return out


# ----------------------------------------------------------------------------------------------------------------------
# SMP training arm (BASELINE.json configs[1])
# ----------------------------------------------------------------------------------------------------------------------
def train_arm(args, dev, world, rank, dist_mod=None, e2e=False, dump=None):
    """ORT supermask training, bf16 tensor-core GEMMs with fp32 master weights + fp32 mask logits, 5 captions/image with the
    encoder run once, Bernoulli masks + dropout + sparsity loss + clip + Adam inside the timed step; at N > 1 the NCCL
    all-reduce of the flat dWm buffer (tests/test_ddp_cpu.py covers the sharding logic).  ``dump``: a dict that receives
    the last timed step's loss and a seeded sample of the weights and mask logits it left."""
    from sparse_caption_b200 import lib
    from sparse_caption_b200 import synthetic
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200.trainer import OrtTrainer
    cfg = ModelCfg(dict(CFG, max_seq_length=17))
    from sparse_caption_b200 import distributed as D
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=0.0, device=dev)
    tr = OrtTrainer(sd, cfg, mask_type="supermask", precision="bf16", device=dev, seed=8888,  # same mask seed on every rank
                    use_graph=not args.no_train_graph, fused_st=not (world > 1 and args.exchange == "sharded"))
    B, S, T = args.train_images, 5, 17
    att, boxes, seqs, masks = _train_batch(B, S, T, CFG["vocab_size"], rank)
    seqs, masks = seqs.pin_memory(), masks.pin_memory()
    opt = dict(lr=3e-4, sparsity_target=0.95, sparsity_weight=30.0, current_step=100, max_step=1000)
    all_reduce = exchange = None
    if world > 1 and args.exchange == "sharded":
        exchange = D.ShardedExchange(device=dev)  # reduce-scatter -> Adam on the owned shard -> all-gather, per bucket
    else:
        all_reduce = D.make_all_reduce(async_op=True)  # NCCL SUM of the gradient buckets each backward phase finishes
    gtok = D.global_token_count(masks.to(dev), T)

    def step():
        return tr.train_step(att, boxes, seqs, masks, seq_per_img=S, all_reduce=all_reduce, exchange=exchange, global_tokens=gtok, **opt)

    def barrier():
        if dist_mod is not None:
            dist_mod.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(3, args.warmup if e2e else 3)):
        step()
    barrier()
    before = lib.launch_count
    n_steps = args.steps if e2e else args.train_steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_steps):
        loss = step()
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    if dump is not None:   # (110 M weights and as many logits: 2^20 of each, the same positions in every run)
        g = torch.Generator().manual_seed(0)
        for name, flat in (("weights_sample", tr.flat_w), ("mask_logits_sample", tr.flat_s)):
            dump[name] = flat[torch.randint(flat.numel(), (1 << 20,), generator=g).to(dev)].cpu().numpy()
        dump["loss"] = loss.detach().double().reshape(1).cpu().numpy()
    launches = (lib.launch_count - before) // n_steps
    # end to end: the same step with the loss read back to the host every step (the reference loop's loss.item(), :142,155)
    host_loss = torch.zeros(1).pin_memory()
    e0.record()
    for _ in range(n_steps):
        host_loss.copy_(step().reshape(1), non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    t = torch.tensor([ms_dev, ms_e2e], device=dev, dtype=torch.float64)
    # every rank's loss is its share of the GLOBAL mean (normalised by the global token count): their sum is the loss
    loss_g = loss.detach().double().reshape(1).clone()
    if dist_mod is not None:
        dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
        dist_mod.all_reduce(loss_g, op=dist_mod.ReduceOp.SUM)
    ms, ms_e = float(t[0]) / n_steps, float(t[1]) / n_steps
    if rank != 0:
        return None
    # GEMM share / tensor roofline from one instrumented step
    lib.profile = []
    tr.use_graph = False  # per-launch event timing needs the eager launch sequence
    tr.train_step(att, boxes, seqs, masks, seq_per_img=S, all_reduce=None, global_tokens=gtok, **opt)  # rank-local
    torch.cuda.synchronize(dev)
    prof, lib.profile = lib.profile, None
    gemm_ms = sum(a.elapsed_time(b) for n, m, a, b in prof if m and m[0] == "gemm_bf16")
    gemm_fl = sum(2.0 * m[1] * m[2] * m[3] for n, m, a, b in prof if m and m[0] == "gemm_bf16")
    tot_ms = sum(a.elapsed_time(b) for n, m, a, b in prof)
    peaks = load_peaks()
    tf_eager = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms else 0.0
    try:
        g_us, g_fl = time_train_gemms(prof, dev)
        tf = g_fl / g_us / 1e6
    except Exception as ex:  # diagnostics only: fall back to the event timing of the eager step
        print(f"in-graph training GEMM timing skipped: {ex}", file=sys.stderr)
        g_us, tf = None, tf_eager
    h2d = att.numel() * 4 + boxes.numel() * 4 + seqs.numel() * 8 + masks.numel() * 4
    return {"metric": "smp_train_images_per_sec", "value": world * B / (ms / 1e3), "unit": "images/s", "n_gpus": world, "ms_per_step": ms,
            "e2e": {"value": world * B / (ms_e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e},
            "collective": "none (1 GPU)" if world == 1 else (
                "per gradient bucket (4 backward phases): NCCL reduce-scatter -> Adam on the owned 1/N shard -> all-gather of the updated "
                "weights + mask logits, on a side stream under the next phase" if exchange is not None else
                "NCCL all-reduce(sum) of the fp32 dWm buckets (gradient w.r.t. the masked weights: 222 MB/step, half of dW + dS; the "
                "straight-through dW / dS are formed inside the optimizer kernel), started after each of the 4 backward phases"),
            "images_per_gpu_per_step": B, "captions_per_image": S, "positions": T, "dtype": "bf16 GEMM / fp32 master+logits",
            "loss": float(loss_g[0]), "loss_note": "global mean over all ranks' tokens (all-reduced)", "gpu_launches_per_step": launches,
            "h2d_bytes_per_step": h2d,
            "includes": "H2D of the batch, Bernoulli masks, dropout, sparsity loss, clip + Adam (2 groups)",
            "algorithmic_gflop_per_step": gemm_fl / 1e9,
            "step_tflops": gemm_fl / (ms / 1e3) / 1e12, "step_frac_of_sustained_peak": gemm_fl / (ms / 1e3) / 1e12 / peaks["tf_sus"],
            "roofline": {"kernel": "sc_gemm_bf16_kernel (fwd + dgrad + wgrad launches of one step, each through its own entry point)",
                         "bound": "tensor", "achieved": tf, "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": tf / peaks["tf_burst"],
                         "traffic": None, "gemm_us_per_step_in_graph": g_us, "achieved_eager_events": tf_eager,
                         "note": "in-graph timing per shape (20 launches, CUDA events); wgrad figures include the split-K reduction kernel",
                         "share_of_step": gemm_ms / tot_ms if tot_ms else None}}


def _claim_stdout():
    """Route everything that libraries print on fd 1 (e.g. NCCL's version banner) to stderr; the returned file object
    is the real stdout, used for the ONE JSON line of the driver contract."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    return real


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="infer", choices=["infer", "train", "acort", "scst"],
                    help="workload: BASELINE.json configs[2] (default; carries configs[1] under `train`), configs[1], configs[3], configs[4]")
    ap.add_argument("--images", type=int, default=0, help="images per GPU per step (0 = the workload's own: 512 / 512 / 1024)")
    ap.add_argument("--backend", default="dense", choices=["dense", "csr", "sell", "auto"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the SMP training arm (BASELINE.json configs[1])")
    ap.add_argument("--train-images", type=int, default=50, help="images per GPU per training step (5 captions each)")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--exchange", default="allreduce", choices=["sharded", "allreduce"],
                    help="data-parallel gradient exchange of the training arm")
    ap.add_argument("--no-train-graph", action="store_true", help="diagnostic: eager launches instead of the captured training graph")
    ap.add_argument("--cpu-images", type=int, default=64)
    ap.add_argument("--ln-fold", action="store_true", help="LayerNorm folded into the consuming GEMMs (sc_linear_ln) instead of separate LayerNorm kernels")
    ap.add_argument("--prefetch", action="store_true", help="e2e arm: H2D of the next batch on a copy stream underneath the previous decode of the same slot")
    ap.add_argument("--no-fuse-topk", action="store_true", help="diagnostic: materialise the logits (sc_linear + sc_beam_step) instead of the fused generator + beam row pass")
    ap.add_argument("--no-pdl", action="store_true", help="diagnostic: disable programmatic dependent launch")
    ap.add_argument("--coalesce", type=int, default=0, help="queued batches the engine decodes as ONE device batch (dynamic batching: the decode "
                         "GEMMs of G batches run as one M = G x rows GEMM); a timed step stays one batch of --images.  0 = the largest of "
                         "5 / 4 / 2 that divides --steps (measured: scripts/gpu_dec_ab4.sh)")
    ap.add_argument("--slots", type=int, default=0, help="device launches in flight (pipeline slots: stream + workspaces + graphs each); 0 = auto")
    ap.add_argument("--e2e-coalesce", type=int, default=0, help="--coalesce of the end-to-end arm (0 = 2 when --steps is even: smaller device batches "
                         "start their H2D copies earlier, so the pipeline of copy -> encode -> decode fills faster)")
    ap.add_argument("--e2e-slots", type=int, default=0, help="--slots of the end-to-end arm (0 = auto)")
    ap.add_argument("--dec-ctas", default="48,60", help="persistent-grid targets of the decode GEMMs in the throughput regime: CTAs for the wide "
                         "(qkv, ff1) and for the N = d_model GEMMs (OrtEngine dec_ctas); 0,0 = one CTA per SM / two tiles per CTA as before")
    ap.add_argument("--e2e-schedule", default="", help="queued batches per launch of the end-to-end arm, e.g. 2,2,4,4,4,4 (sums to --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="after the timed steps, write what the timed path returned for its "
                         "last step as DIR/<name>.npy (float32 / float64, at most 64 MB, rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.config == "train":
        return train_main(args, out, rank, local_rank, world)

    wl = WORKLOADS[args.config]
    if args.images <= 0:
        args.images = wl["images"]
    if args.coalesce <= 0:
        cands = (2,) if args.config == "scst" else (5, 4, 2)   # (scst: 1024 images and two decodes per step already)
        args.coalesce = next((g for g in cands if args.steps % g == 0), 1)
    if args.slots <= 0:
        # the K / G device launches go round-robin over the slots (stream + workspaces + graphs each); a slot count that divides
        # them keeps every round of the pipeline full, long runs amortise fill / drain anyway
        launches = max(1, args.steps // max(1, args.coalesce))
        args.slots = next((sl for sl in (4, 3, 2) if launches % sl == 0), min(4, launches)) if args.coalesce > 1 else (
            8 if args.steps >= 24 else next((sl for sl in (8, 7, 6, 5, 4) if args.steps % sl == 0), 4))
    cfgd = wl["cfg"]
    L = cfgd["max_seq_length"]
    beams = [int(o.get("beam_size", 1)) for o in wl["decodes"]]
    config = {"workload": f"{wl['label']} ({args.images} images/GPU/step) [BASELINE.json configs[{wl['idx']}]]",
              "images_per_gpu_per_step": args.images, "beam": beams if len(beams) > 1 else beams[0], "max_len": L, "sparsity": wl["sparsity"],
              "sharding": f"images by rank x{world}, no data-path collective", "decoder_gemm_backend": args.backend,
              "batches_in_flight": args.slots * max(1, args.coalesce), "coalesced_batches_per_launch": max(1, args.coalesce),
              "l2_policy": f"inputs_larger_than_L2 ({args.images * N_BOX * 2048 * 4 / 1e6:.0f} MB fresh fp32 features + ~0.7 GB of activations/KV per step vs 126 MB L2)"}

    if args.impl == "reference":
        if rank != 0:
            return
        # K timed steps and W warm-up steps as asked; one step = a BOUNDED SAMPLE of the workload's step (--cpu-images images
        # instead of --images: ~0.6 s on 16 cores) - stated in `config` - so the default K=10 / W=3 run takes ~10 s
        warm = max(1, args.warmup)
        steps = max(1, args.steps)
        v, spp, cores = cpu_arm(steps, warm, args.cpu_images, wl)
        config = dict(config, images_per_gpu_per_step=args.cpu_images, sampled_from_images_per_step=args.images, batches_in_flight=1,
                      coalesced_batches_per_launch=1,
                      workload=config["workload"] + f" - reference arm: bounded sample of {args.cpu_images} images per step")
        print(json.dumps({"impl": "reference", "metric": wl["metric"], "value": v, "unit": wl["unit"], "n_gpus": args.gpus, "steps": steps,
                          "warmup": warm, "ms_per_step": spp * 1e3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": wl["unit"], "cores": cores, "kind": "port",
                                           "sample": f"{steps} x {args.cpu_images} images, same model/beam/length, torch fp32 on host cores"},
                          "e2e": {"value": v, "unit": wl["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), file=out, flush=True)
        return

    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from sparse_caption_b200 import lib, synthetic
    from sparse_caption_b200.engine import ModelCfg, OrtEngine
    lib.load()
    if args.no_pdl:
        from sparse_caption_b200 import kernels as _K
        _K.set_pdl(False)
    cfg = ModelCfg(cfgd)
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=wl["sparsity"], device=dev)
    G = max(1, args.coalesce)
    assert args.steps % G == 0, "--steps must be a multiple of --coalesce"
    # >= 8 batches in flight (throughput regime): the decode GEMMs run 256-wide tiles on persistent grids of ~48 CTAs (qkv, ff1:
    # 8 - 10 tiles per CTA) / ~60 CTAs (the N = d_model GEMMs), sized per workspace by the engine (OrtEngine dec_ctas)
    dec_ctas = tuple(int(v) for v in args.dec_ctas.split(",")) if args.slots * G >= 8 else None
    dec_tiles = None
    if dec_ctas is not None and not any(dec_ctas):   # (the round-2 start configuration, kept for A/B runs)
        dec_ctas, dec_tiles = None, {k: 20003256 for k in ("qkv", "o", "cq", "co", "ff1", "ff2")}
    eng = OrtEngine(sd, cfg, precision="bf16", sparse_backend=args.backend, device=dev, ln_fold=args.ln_fold,
                    fuse_topk=not args.no_fuse_topk, dec_ctas=dec_ctas, dec_tiles=dec_tiles)
    B = args.images * G      # device batch = G queued batches of --images
    F = cfgd["att_feat_size"]
    # two distinct pinned host batches, alternated
    host = [synthetic.synthetic_inputs(B, N_BOX, F, seed=8888 + rank + 100 * i, pin=True) for i in range(2)]
    opts = wl["decodes"]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident arm: inputs already in HBM ----------------
    # `slots` device launches are in flight at once: slot s = its own stream, workspaces and CUDA graphs (engine.submit);
    # every timed step is still one full batch of --images (encoder + all decode steps + beam bookkeeping).
    S = max(1, args.slots)
    slots = list(range(1, S + 1))
    cur = torch.cuda.current_stream(dev)
    encs = {}
    for s in slots:
        # inputs resident in HBM (fp32, as the data loader delivers them) -> the slot's workspaces + graphs
        eng.submit(host[s & 1][0].to(dev), host[s & 1][1].to(dev), None, opts, slot=s)
        encs[s] = eng._get_enc_ws(B, N_BOX, False, s)
    eng.wait(host=True)
    torch.cuda.synchronize(dev)
    launches_per_call = encs[slots[0]].launches + sum(eng._get_dec_ws(B, b, N_BOX, b == 1, slots[0]).launches for b in beams)

    def dev_step(i):
        s = slots[i % S]
        with torch.cuda.stream(eng.stream(s)):
            eng.run_encoder(encs[s])
            return [eng.decode(encs[s], o) for o in opts]

    def fork():
        for s in slots:
            eng.stream(s).wait_stream(cur)

    def join():
        for s in slots:
            cur.wait_stream(eng.stream(s))

    n_warm, n_timed = max(1, -(-args.warmup // G)), args.steps // G   # device launches (each = G steps of --images images)
    fork()
    for i in range(n_warm):
        dev_step(i)
    join()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:  # one nvidia-smi poller per job, not per rank
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fork()
    for i in range(n_timed):
        last = dev_step(i)
    join()
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    dump = None
    if args.dump_outputs and rank == 0:
        # (seq, log-probs) [B, beam, L] per decode of the last timed launch (its G coalesced batches), views of the slot's
        # workspaces: copied now, outside the timed region; the beam size names the decode (scst: beam 5 and greedy, beam 1)
        dump = {}
        for (seq, lp), b in zip(last, beams):
            dump[f"beam{b}_seq"], dump[f"beam{b}_logprobs"] = seq.cpu().numpy(), lp.cpu().numpy()

    # ---------------- end-to-end arm: pinned host inputs -> tokens on the host ----------------
    # --e2e-coalesce 0 (default): 4 queued batches per launch when --steps allows it (else 2 / 1).  The H2D copy of a launch's
    # batches paces its start (3 ms per batch over PCIe): measured schedules for 20 steps (scripts/gpu_e2e_sched.sh, ms/step):
    # 10 x 2: 6.00, 5 x 4: 5.89, 2,2,4,4,4,4: 5.87, 2,3,5,5,5: 5.85, 4 x 5: 5.97, ramp 1,1,2,4,4,4,4: 6.54 (its single-batch
    # launches are latency-bound chains that leave the SMs idle)
    if args.e2e_schedule:
        sched = [int(g) for g in args.e2e_schedule.split(",")]
        assert sum(sched) == args.steps, "--e2e-schedule must sum to --steps"
    else:
        ge = args.e2e_coalesce if args.e2e_coalesce > 0 else next(g for g in (4, 2, 1) if args.steps % g == 0 and g <= max(1, G))
        assert args.steps % ge == 0, "--steps must be a multiple of --e2e-coalesce"
        sched = [ge] * (args.steps // ge)
    Ge = max(sched)
    ne_timed = len(sched)
    Se = args.e2e_slots if args.e2e_slots > 0 else min(5, ne_timed)
    eslots = list(range(101, 101 + Se))
    Bmax = args.images * Ge
    big = host if Bmax <= B else [synthetic.synthetic_inputs(Bmax, N_BOX, F, seed=8888 + rank + 100 * i, pin=True) for i in range(2)]
    outs = {}   # (slot index, batches in the launch) -> pinned result buffers per decode

    def e2e_run(batches):
        def e2e_step(i):
            g = sched[i]
            att, boxes = batches[i & 1]
            k = i % Se
            if (k, g) not in outs:
                outs[(k, g)] = [(torch.empty(args.images * g, max(b, 1), L, dtype=torch.int32).pin_memory(),
                                 torch.empty(args.images * g, max(b, 1), L, dtype=torch.float32).pin_memory()) for b in beams]
            eng.submit(att[: args.images * g], boxes[: args.images * g], None, opts, slot=eslots[k], out=outs[(k, g)], prefetch=args.prefetch)
        for i in range(ne_timed):  # one untimed pass of the schedule: every (slot, batch size) pair's workspaces / graphs are warm
            e2e_step(i)
        eng.wait()
        barrier()
        e0.record()
        for i in range(ne_timed):
            e2e_step(i)
        eng.wait()
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    ms_e2e = e2e_run(big)
    # the same with bf16 pinned host features (half the H2D bytes; the engine lands them directly in the GEMM operand buffer)
    host16 = [(a.to(torch.bfloat16).pin_memory(), b) for a, b in big]
    ms_e2e16 = e2e_run(host16)
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)
    per_img = big[0][0][0].numel()
    h2d = args.images * (per_img * 4 + N_BOX * 4 * 4)     # per step of --images: fp32 features + boxes
    h2d16 = args.images * (per_img * 2 + N_BOX * 4 * 4)
    d2h = sum(args.images * max(b, 1) * L * 8 for b in beams)   # tokens (int32) + log-probs (fp32)
    del host16

    t = torch.tensor([ms_dev, ms_e2e, ms_e2e16], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_e2e16 = float(t[0]), float(t[1]), float(t[2])
    per_s = lambda ms: world * args.images * args.steps / (ms / 1e3)
    value, e2e_value = per_s(ms_dev), per_s(ms_e2e)

    train = None
    if not args.no_train and args.config == "infer":
        train = train_arm(args, dev, world, rank, dist_mod=dist)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- roofline leg: one instrumented step without graphs ----------------
    peaks = load_peaks()
    traffic = load_traffic()
    # the DEVICE batch of the timed region (G coalesced batches of --images): the roofline is quoted on the shapes that were launched
    Bp = B
    att_p, box_p = host[0][0][:Bp], host[0][1][:Bp]
    eng2 = OrtEngine(sd, cfg, precision="bf16", sparse_backend=args.backend, device=dev, use_graphs=False,
                     ln_fold=args.ln_fold, fuse_topk=not args.no_fuse_topk, dec_ctas=dec_ctas, dec_tiles=dec_tiles)
    enc2 = eng2.encode(att_p, box_p)
    for o in opts:
        eng2.decode(enc2, o)
    torch.cuda.synchronize(dev)
    lib.profile = []
    eng2.run_encoder(enc2)
    for o in opts:
        eng2.decode(enc2, o)
    torch.cuda.synchronize(dev)
    prof, lib.profile = lib.profile, None
    by = {}
    for name, meta, a, b in prof:
        key = meta[0] if meta else name
        d = by.setdefault(key, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0})
        d["ms"] += a.elapsed_time(b)
        d["n"] += 1
        if meta and meta[0].startswith("gemm"):
            _, M, N, Kd, xs, wsz, ys = meta[:7]
            d["flops"] += 2.0 * M * N * Kd
            d["bytes"] += M * Kd * xs + N * Kd * wsz + M * N * ys
        elif meta and meta[0] in ("csr_spmm", "sell_spmm"):
            _, M, N, Kd, xs, nnz, ys = meta
            d["flops"] += 2.0 * M * nnz
            d["bytes"] += M * Kd * xs + nnz * (xs + 2) + M * N * ys
    total_ms = sum(d["ms"] for d in by.values())
    top = max(by, key=lambda k: by[k]["ms"])
    g = by.get("gemm_bf16", by[top])
    # The per-launch events above include the host's launch gaps (eager ctypes launches): they give the kernel's SHARE of
    # the step.  The duration behind `achieved` is measured without them: every GEMM shape of the step, 40 launches inside
    # one CUDA graph on the current stream, CUDA events around two replays.
    shapes = {}
    for name, meta, a, b in prof:
        if meta and meta[0] == "gemm_bf16":
            key = tuple(meta[1:7]) + tuple(meta[8:10]) + ((meta[10] if len(meta) > 10 else 0),)   # (+ the engine's tile hint)
            shapes[key] = shapes.get(key, 0) + 1
    from sparse_caption_b200 import kernels as KK
    topk_beam = max([b for b in beams if b > 1] or [3])

    def make_run(M, N, Kd, ys, has_res, relu, tile, nbuf):
        x = torch.randn(M, Kd, device=dev).bfloat16()
        w = torch.randn(N, Kd, device=dev).bfloat16()
        bias = torch.randn(N, device=dev)
        if ys == 0:  # generator fused with the beam row pass: no output tile, 12-float records per (row, tile half)
            part = torch.empty(M, KK.linear_topk_parts(N), 12, device=dev)
            return lambda i: KK.linear_topk(x, w, bias, part, candidates=min(5, topk_beam))
        outs_ = [torch.empty(M, N, device=dev, dtype=torch.bfloat16 if ys == 2 else torch.float32) for _ in range(nbuf)]
        if has_res:  # the engine's residual GEMMs update the fp32 residual stream in place
            return lambda i: KK.linear(x, w, bias, residual=outs_[i % nbuf], relu=relu, out=outs_[i % nbuf], tile_n=tile)
        return lambda i: KK.linear(x, w, bias, relu=relu, out=outs_[i % nbuf], tile_n=tile)

    gemm_us, gemm_fl, dom = 0.0, 0.0, None
    for (M, N, Kd, xs, wsz, ys, has_res, relu, tile), cnt in shapes.items():
        us = _time_graph(make_run(M, N, Kd, ys, has_res, relu, tile, 4), dev)
        gemm_us += us * cnt
        gemm_fl += 2.0 * M * N * Kd * cnt
        if dom is None or us * cnt > dom[0]:
            dom = (us * cnt, M, N, Kd, us, cnt, xs * M * Kd + wsz * N * Kd + ys * M * N + (4 * M * N if has_res else 0), ys, has_res)
    # the same shapes with several streams running them concurrently - the regime of the timed region (launches in flight):
    # microseconds of wall time per GEMM = elapsed / (streams * launches)
    conc_us, conc_fl = 0.0, 0.0
    CS = max(2, min(8, S if G > 1 else S * G))   # device launches in flight in the timed region
    try:
        streams = [torch.cuda.Stream(dev) for _ in range(CS)]
        cur_s = torch.cuda.current_stream(dev)
        for (M, N, Kd, xs, wsz, ys, has_res, relu, tile), cnt in shapes.items():
            graphs = []
            for st in streams:
                run = make_run(M, N, Kd, ys, has_res, relu, tile, 2)
                run(0)
                torch.cuda.synchronize(dev)
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    for i in range(20):
                        run(i)
                graphs.append((gr, run))

            def go():
                for st, (gr, _) in zip(streams, graphs):
                    st.wait_stream(cur_s)
                    with torch.cuda.stream(st):
                        gr.replay()
                        gr.replay()
                for st in streams:
                    cur_s.wait_stream(st)
            go()
            torch.cuda.synchronize(dev)
            e0.record(); go(); e1.record()
            torch.cuda.synchronize(dev)
            us = e0.elapsed_time(e1) * 1e3 / (CS * 40)
            conc_us += us * cnt
            conc_fl += 2.0 * M * N * Kd * cnt
            del graphs
    except Exception as ex:  # diagnostics only
        print(f"concurrent GEMM timing skipped: {ex}", file=sys.stderr)
    tf_conc = conc_fl / conc_us / 1e6 if conc_us else None
    tf = gemm_fl / gemm_us / 1e6 if gemm_us else 0.0
    tf_dom = 2.0 * dom[1] * dom[2] * dom[3] / dom[4] / 1e6 if dom else 0.0
    dom_key = None if dom is None else f"{dom[1]},{dom[2]},{dom[3]},{dom[7]},{int(bool(dom[8]))}"
    try:
        hbm = hbm_kernel_roofline(dev, Bp, topk_beam, N_BOX, cfgd, peaks)
    except Exception as ex:
        print(f"HBM kernel timing skipped: {ex}", file=sys.stderr)
        hbm = None
    step_tf = (gemm_fl / G) / (ms_dev / args.steps / 1e3) / 1e12   # (gemm_fl covers one device launch = G steps)
    roofline = {"kernel": "sc_gemm_bf16_kernel (tcgen05/TMEM/TMA; every GEMM launch of one step)", "bound": "tensor", "achieved": tf,
                "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": tf / peaks["tf_burst"],
                # dram__bytes_read.sum + dram__bytes_write.sum per launch of THE SHAPE REPORTED as dominant, from the committed ncu
                # capture keyed by shape (profiles/r02_gemm_traffic.json; cold-cache capture, one launch) - null when not captured
                "traffic": traffic.get(dom_key) if dom_key else None, "traffic_key": dom_key,
                "peak_source": f"{peaks['src']} MEASURED_PEAKS.json bf16_tflops (burst: shapes timed alone, in-graph)",
                "achieved_in_flight": tf_conc, "frac_in_flight": (tf_conc / peaks["tf_sus"]) if tf_conc else None,
                "in_flight_note": f"same shapes, {CS} streams concurrently (the timed region's regime), wall time per GEMM; vs sustained peak",
                "whole_step_tflops": step_tf, "whole_step_frac_of_sustained_peak": step_tf / peaks["tf_sus"],
                "device_batch_images": Bp, "steps_per_device_launch": G,
                "launches": g["n"], "avg_launch_us": gemm_us / max(1, g["n"]),
                "launches_note": "GEMM launches of ONE device launch (G coalesced steps), timed at the shapes and tile hints the timed region uses",
                "algorithmic_gflop_per_step": gemm_fl / G / 1e9,
                "dominant_shape": None if dom is None else {"M": dom[1], "N": dom[2], "K": dom[3], "launches": dom[5], "us_per_launch": dom[4],
                                                            "tflops": tf_dom, "algorithmic_bytes": dom[6],
                                                            "hbm_floor_us": dom[6] / (peaks["hbm"] * 1e3)},
                "share_of_step": g["ms"] / total_ms if total_ms else None,
                "share_source": "per-launch CUDA events of one un-graphed step (host launch gaps included); the ncu launch list "
                                "profiles/r02c_infer_launches_summary.txt (kernels of the same command) gives the same share",
                "kernel_time_breakdown_ms": {k: round(v["ms"], 3) for k, v in sorted(by.items(), key=lambda kv: -kv[1]["ms"])},
                "hbm_kernels": hbm}

    cpu = None
    if not args.no_cpu_baseline and world == 1:  # (rank 0 at N = 1 only; at N > 1 the driver reads it from the N = 1 line)
        # bounded sample of ~10-20 s of CPU work: rate from one 64-image pass, then one pass sized from it
        v0, _, cores = cpu_arm(1, 1, args.cpu_images, wl)
        n_img = int(min(1024, max(args.cpu_images, 32 * round(v0 * 12 / 32))))
        v, spp, cores = cpu_arm(1, 0, n_img, wl)
        cpu = {"value": v, "unit": wl["unit"], "cores": cores, "kind": "port", "seconds": spp,
               "sample": f"1 x {n_img} images (same model, beams {beams}, L={L}; sized for ~12 s), torch fp32 oracle port of the reference path on host cores"}

    line = {"metric": wl["metric"], "value": value, "unit": wl["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_value, "unit": wl["unit"], "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "host_features": "fp32 pinned (the reference loader's dtype)",
                    "batches_per_launch_schedule": sched, "launches_in_flight": Se},
            "e2e_bf16_host": {"value": per_s(ms_e2e16), "unit": wl["unit"], "h2d_bytes_per_step": h2d16, "d2h_bytes_per_step": d2h,
                              "ms_per_step": ms_e2e16 / args.steps, "host_features": "bf16 pinned"},
            "gpu_launches": launches_per_call * n_timed, "clocks": sampler.summary(), "roofline": roofline,
            "cpu_baseline": cpu, "train": train}
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    print(json.dumps(line), file=out, flush=True)
    if dist is not None:
        dist.destroy_process_group()


def train_main(args, out, rank, local_rank, world):
    """--config train: the SMP training arm (BASELINE.json configs[1]) as the line's own metric."""
    config = {"workload": f"ORT 6x512 supermask (SMP) training, bf16 GEMMs / fp32 master weights + mask logits, {args.train_images} images x 5 "
                          f"captions per GPU per step, T=17, V=10000, encoder once per image [BASELINE.json configs[1]]",
              "images_per_gpu_per_step": args.train_images, "captions_per_image": 5, "positions": 17,
              "sharding": (f"images by rank x{world}; NCCL all-reduce of dWm (the weights' and mask logits' gradients follow from it)"
                           if world > 1 else "1 GPU"),
              "l2_policy": "inputs_larger_than_L2 (443 MB of weights + logits, 0.9 GB of saved activations per step vs 126 MB L2)"}
    if args.impl == "reference":
        if rank != 0:
            return
        n_img = min(args.train_images, 10)
        steps, warm = max(1, args.steps), max(1, min(args.warmup, 1))
        v, spp, cores = cpu_train_arm(steps, warm, n_img)
        config = dict(config, images_per_gpu_per_step=n_img, sampled_from_images_per_step=args.train_images,
                      workload=config["workload"] + f" - reference arm: bounded sample of {n_img} images per step")
        print(json.dumps({"impl": "reference", "metric": "smp_train_images_per_sec", "value": v, "unit": "images/s", "n_gpus": args.gpus,
                          "steps": steps, "warmup": warm, "ms_per_step": spp * 1e3, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                                           "sample": f"{steps} x {n_img} images x 5 captions, forward + backward + clip + Adam, torch fp32 autograd over the oracle"},
                          "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), file=out, flush=True)
        return
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from sparse_caption_b200 import lib
    lib.load()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dump = {} if args.dump_outputs and rank == 0 else None
    tr = train_arm(args, dev, world, rank, dist_mod=dist, e2e=True, dump=dump)
    sampler.stop_flag = True
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    sampler.join(timeout=2)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        v, spp, cores = cpu_train_arm(3, 1, 10)
        cpu = {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "seconds": spp * 3,
               "sample": "3 x 10 images x 5 captions (forward + backward + clip + Adam), torch fp32 autograd over the oracle port on host cores"}
    line = {"metric": tr["metric"], "value": tr["value"], "unit": tr["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": tr["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config, "e2e": tr["e2e"], "gpu_launches": tr["gpu_launches_per_step"] * args.steps,
            "clocks": sampler.summary(), "roofline": tr["roofline"], "cpu_baseline": cpu,
            "train_detail": {k: v for k, v in tr.items() if k not in ("roofline", "e2e")}}
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    print(json.dumps(line), file=out, flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
