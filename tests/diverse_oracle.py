"""CPU restatement of diverse beam search (batch_beam_search with group_size > 1, caption_model.py:30-226; paths relative
to the reference checkout), built on the pinned oracle (oracle/ort_oracle.py: DecodeState, decode_step, beam_select,
length_penalty).  TEST INFRASTRUCTURE ONLY: the checker of the diverse-beam kernels, engine and model surface.

With diversity_lambda = 0 every group is an independent width-bdash beam search, so tests/test_diverse_beam_cpu.py pins
this restatement group by group to the reference goldens of the group-size-1 search."""
from typing import List, Tuple

import torch

from oracle.ort_oracle import SD, Cfg, DecodeState, Tensor, beam_select, decode_step, length_penalty


def add_diversity(beam_seq_table: List[Tensor], logprobs: Tensor, local_t: int, group: int, diversity_lambda: float,
                  bdash: int) -> Tuple[Tensor, Tensor]:
    """caption_model.py:33-52.  Returns (augmented, unaugmented) log-probs: the augmented ones are lowered by lambda per beam
    of an earlier group whose token at position ``local_t`` of its CURRENT history is that word (duplicates count twice).
    The earlier groups have already stepped in this global step, so their histories are reordered up to their own (later)
    local step - which is why the groups cannot be run in lockstep."""
    unaug = logprobs.clone()
    if group == 0:
        return logprobs, unaug
    B = beam_seq_table[0].shape[0]
    change = logprobs.new_zeros(B, logprobs.shape[-1])
    for p in range(group):
        prev = beam_seq_table[p][:, :, local_t]  # [B, bdash]
        for j in range(bdash):
            change.scatter_add_(1, prev[:, j].unsqueeze(-1), change.new_ones(B, 1))
    if local_t == 0:  # one row per image (only beam 0 is expanded)
        return logprobs - change * diversity_lambda, unaug
    return logprobs - change.repeat_interleave(bdash, 0) * diversity_lambda, unaug


def diverse_groups(opt: dict) -> Tuple[int, int, float]:
    """(G, bdash, lambda) of the decode options (caption_model.py:114-123): bdash = beam_size // group_size beams per group."""
    beam, G = int(opt.get("beam_size", 10)), int(opt.get("group_size", 1))
    return G, beam // G, float(opt.get("diversity_lambda", 0.5))


def diverse_beam_core(init_logprobs: Tensor, advance, B: int, V: int, L: int, eos: int, pad: int, opt: dict,
                      margins: Tensor = None):
    """The group schedule and bookkeeping of batch_beam_search (caption_model.py:126-226) over a log-prob source.

    ``init_logprobs`` [B, V]: the BOS step's log-probs (every group starts from them, not tempered).
    ``advance(group, state_ix, it, local_t)``: reorder the group's state with ``state_ix`` [B*bdash], feed tokens ``it``
    [B*bdash] and return the next log-probs [B*bdash, V] (already ``log_softmax(lp / T)``, :214-218).  Tests drive this with
    scripted log-probs, the model with ``decode_step``.

    Global step t = 0 .. L+G-2; group g runs at local step t - g when 0 <= t - g <= L-1, groups in ascending order.  The
    running sum takes the AUGMENTED log-prob (so does the finished score p), the stored per-token log-prob the unaugmented
    one.  Returns (seq [B, G*bdash, L], logps [B, G*bdash, L], p [B, G*bdash], done [B][G*bdash] dicts {seq, logps,
    unaug_p, p}): each group's finished beams sorted stably by -p, the first bdash kept, groups concatenated in order.
    ``margins`` (optional fp32 [B, G], filled in place): per image and group the smallest score gap of any decision that
    group made (consecutive entries of its sorted candidate list down to the first rejected one, every step; consecutive
    entries of its final ranking), as ``oracle.ort_oracle.beam_search`` records for group_size 1."""
    G, bdash, lam = diverse_groups(opt)
    constraint = opt.get("decoding_constraint", 0)
    # remove_bad_endings / suppress_UNK as the model surface passes them (the ids of model.bad_endings_ix, and the last
    # column when the vocabulary calls it UNK)
    bad = torch.tensor(sorted(opt["bad_endings_ix"])) if opt.get("bad_endings_ix") else None
    pen_col = int(opt.get("penalized_col", -1))
    pen = length_penalty(opt.get("length_penalty", ""))
    seq_t = [torch.zeros(B, bdash, 0, dtype=torch.long) for _ in range(G)]
    lp_t = [torch.zeros(B, bdash, 0) for _ in range(G)]
    sum_t = [torch.zeros(B, bdash) for _ in range(G)]
    logprobs_t = [init_logprobs.clone() for _ in range(G)]
    done: List[List[List[dict]]] = [[[] for _ in range(G)] for _ in range(B)]
    for t in range(L + G - 1):
        for g in range(G):
            tau = t - g
            if not 0 <= tau <= L - 1:
                continue
            logprobs = logprobs_t[g].clone()
            if constraint and tau > 0:
                logprobs.scatter_(1, seq_t[g][:, :, tau - 1].reshape(-1, 1), float("-inf"))
            if bad is not None and tau > 0:                                                     # :161-168
                logprobs[torch.isin(seq_t[g][:, :, tau - 1].reshape(-1), bad), 0] = float("-inf")
            if pen_col >= 0:                                                                    # :169-170
                logprobs[:, pen_col] = logprobs[:, pen_col] - 1000
            aug, unaug = add_diversity(seq_t, logprobs, tau, g, lam, bdash)
            parent, word, new_sum = beam_select(aug, sum_t[g], bdash, first=(tau == 0))     # beam_step, :56-111
            nb = aug.size(0) // B
            if margins is not None:
                s0 = sum_t[g][:, :1] if tau == 0 else sum_t[g]
                top = torch.topk((s0.unsqueeze(-1) + aug.view(B, nb, V)).reshape(B, -1), bdash + 1, dim=-1).values
                margins[:, g] = torch.minimum(margins[:, g], (top[:, :-1] - top[:, 1:]).min(-1).values)
            chosen = unaug.view(B, nb, V).gather(1, parent.unsqueeze(-1).expand(-1, -1, V)).gather(2, word.unsqueeze(-1)).squeeze(-1)
            if tau > 0:
                seq_t[g] = seq_t[g].gather(1, parent.unsqueeze(-1).expand_as(seq_t[g]))
                lp_t[g] = lp_t[g].gather(1, parent.unsqueeze(-1).expand_as(lp_t[g]))
            seq_t[g] = torch.cat([seq_t[g], word.unsqueeze(-1)], -1)
            lp_t[g] = torch.cat([lp_t[g], chosen.unsqueeze(-1)], -1)
            sum_t[g] = new_sum.clone()
            state_ix = (parent + torch.arange(B).unsqueeze(-1) * nb).reshape(-1)
            for b in range(B):                                                                 # :188-210
                is_end = seq_t[g][b, :, tau] == eos
                if tau == L - 1:
                    is_end = torch.ones_like(is_end)
                for v in range(bdash):
                    if is_end[v]:
                        done[b][g].append({"seq": seq_t[g][b, v].clone(), "logps": lp_t[g][b, v].clone(),
                                           "unaug_p": float(lp_t[g][b, v].sum()), "p": pen(tau + 1, float(sum_t[g][b, v]))})
                sum_t[g][b, is_end] -= 1000
            logprobs_t[g] = advance(g, state_ix, seq_t[g][:, :, tau].reshape(-1), tau)
    W = G * bdash
    seq = torch.full((B, W, L), pad, dtype=torch.long)
    seq_lp = torch.zeros(B, W, L)
    done_p = torch.zeros(B, W)
    out = []
    for b in range(B):                                                                         # :221-225
        ranked = [sorted(done[b][g], key=lambda d: -d["p"]) for g in range(G)]
        if margins is not None:
            for g in range(G):
                for v in range(min(bdash, len(ranked[g]) - 1)):
                    margins[b, g] = min(float(margins[b, g]), ranked[g][v]["p"] - ranked[g][v + 1]["p"])
        beams = sum((r[:bdash] for r in ranked), [])
        for v, d in enumerate(beams):
            n = d["seq"].numel()
            seq[b, v, :n] = d["seq"]
            seq_lp[b, v, :n] = d["logps"]
            done_p[b, v] = d["p"]
        out.append(beams)
    return seq, seq_lp, done_p, out


def diverse_beam_search(sd: SD, cfg: Cfg, memory: Tensor, src_mask: Tensor, opt: dict, no_history: bool = False,
                        margins: Tensor = None):
    """batch_beam_search with group_size > 1 (caption_model.py:30-226) over the model: one DecodeState per group, each a
    copy of the state after the shared BOS step (:133-135).  Returns (seq, seq_logprobs, done_p) as ``beam_search``."""
    G, bdash, _ = diverse_groups(opt)
    temperature = opt.get("temperature", 1.0)
    B, L, V = memory.size(0), cfg.max_seq_length, cfg.vocab_size
    st0 = DecodeState(cfg)
    it = torch.full((B,), cfg.bos_token_id, dtype=torch.long)
    logprobs = decode_step(sd, cfg, st0, it, memory, src_mask, no_history)
    states = []
    for _ in range(G):
        s = DecodeState(cfg)
        s.self_k, s.self_v, s.cross_k, s.cross_v = dict(st0.self_k), dict(st0.self_v), dict(st0.cross_k), dict(st0.cross_v)
        s.t = st0.t
        states.append(s)
    memory_r = memory.repeat_interleave(bdash, 0)
    mask_r = src_mask.repeat_interleave(bdash, 0)

    def advance(g, state_ix, it, tau):
        states[g].reorder(state_ix)
        lp = decode_step(sd, cfg, states[g], it, memory_r, mask_r, no_history)
        return torch.log_softmax(lp / temperature, dim=-1)

    seq, seq_lp, done_p, _ = diverse_beam_core(logprobs, advance, B, V, L, cfg.eos_token_id, cfg.pad_token_id, opt, margins)
    return seq, seq_lp, done_p


