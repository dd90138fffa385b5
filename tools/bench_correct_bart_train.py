"""Throughput of CorrectBart fine-tuning on the device (engine.Seq2SeqTrainer, DESIGN.md §3.13).

Workload: the bart-base-chinese shape (6 + 6 layers, d_model 768, FFN 3 072, vocab 21 128), random init, the
C2 (hyp_1, ref) pairs of synth.make_nbest(7176, 10) in batches of 32 and of 256 sentences, dropout 0.1,
mode 1 (forward, backward, AdamW).  Each batch shape runs eagerly once and is captured on its second
occurrence, so the timed pass, a third pass over the same batches, is all graph replays.  For orientation
only: one fp32 autograd step of transformers on the host cores for a small batch.  Writes
profiles/correct_bart_train_bench.json (or --out) with the GPU name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_correct_bart import gpu_context  # noqa: E402


def step_gemm_flops(B, Te, Td, H=768, Ie=3072, Id=3072, Le=6, Ld=6, Vp=21248):
    """Algorithmic GEMM FLOPs of one training step (mode 1) from the shapes: the forward GEMMs, and the dgrad
    and wgrad of each, which cost as much again each (3x).  Encoder row: Q, K, V, out (4 H^2) and the FFN
    (2 H Ie), times 2 FLOPs per MAC; cross K|V of every decoder layer over the encoder rows (2 H^2 per layer);
    decoder row: self Q, K, V, out and cross Q, out (6 H^2) and the FFN (2 H Id); LM head H Vp per decoder row.
    Attention score / context products run outside the GEMMs and are not counted."""
    enc = B * Te * Le * 2 * (4 * H * H + 2 * H * Ie)
    ckv = B * Te * Ld * 2 * (2 * H * H)
    dec = B * Td * Ld * 2 * (6 * H * H + 2 * H * Id)
    head = B * Td * 2 * H * Vp
    return 3.0 * (enc + ckv + dec + head)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=7176)
    ap.add_argument("--batches", type=int, default=16, help="batches per size in the timed pass")
    ap.add_argument("--sizes", default="32,256")
    ap.add_argument("--host-batch", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    a.out = a.out or os.path.join(ROOT, "profiles", "correct_bart_train_bench.json")
    import torch
    from asr_rescoring_b200 import engine, synth
    from asr_rescoring_b200.CorrectBart.train import batch_capacity, make_batches
    from asr_rescoring_b200.tokenizer import SyntheticCharTokenizer
    from oracle import bart_oracle as bo
    from oracle import bart_train_oracle as bto

    cfg = bo.bart_config(d_model=768, layers=6, ffn=3072, vocab=21128, max_position=512)
    cfg.dropout = 0.1
    m = bo.make_model(cfg, seed=5, perturb=False)
    sd = m.state_dict()
    nb = synth.make_nbest(a.utts, 10, seed=0)
    tok = SyntheticCharTokenizer()
    hyps, refs = [hs[0] for hs in nb.hyps], list(nb.refs)
    res = dict(gpu=gpu_context(), workload=dict(shape="bart-base-chinese (6+6, 768, 3072, 21128)", init="random",
                                                pairs=f"C2 (hyp_1, ref), make_nbest({a.utts}, 10)", dropout=0.1,
                                                mode=1), runs=[])
    for S in [int(x) for x in a.sizes.split(",")]:
        batches = make_batches(tok, hyps, refs, S)[:a.batches]
        mb, me, md = batch_capacity(batches)
        with engine.Seq2SeqTrainer(sd, cfg.to_dict(), device=0, lr=1e-5, max_batch=mb, max_enc_len=me,
                                   max_dec_len=md) as tr:
            for _ in range(2):                                   # eager, then capture (+ first replay)
                for b in batches:
                    tr.step(b["input_ids"], b["attention_mask"], b["labels"], mode=1)
            torch.cuda.synchronize()
            l0, r0 = tr.kernel_launches(), tr.graph_replays()
            t0 = time.perf_counter()
            for b in batches:                                    # step() ends in a stream synchronise
                tr.step(b["input_ids"], b["attention_mask"], b["labels"], mode=1)
            dt = time.perf_counter() - t0
            launches, replays = tr.kernel_launches() - l0, tr.graph_replays() - r0
            ws = tr.workspace_bytes()
        n = len(batches)
        sents = sum(b["input_ids"].shape[0] for b in batches)
        tgt = int(sum((b["labels"] != -100).sum() for b in batches))
        flops = sum(step_gemm_flops(b["input_ids"].shape[0], b["input_ids"].shape[1], b["labels"].shape[1])
                    for b in batches)
        run = dict(sents_per_batch=S, steps=n, replays=int(replays), ms_per_step=1e3 * dt / n, sentences_per_s=sents / dt,
                   target_tokens_per_s=tgt / dt, launches_per_step=launches / n, gemm_tflops_per_step=flops / n / 1e12,
                   achieved_gemm_tflop_s=flops / dt / 1e12, workspace_gb=ws / 1e9, capacity=[mb, me, md])
        print(json.dumps(run))
        res["runs"].append(run)
    # orientation: one fp32 autograd step on the host cores
    hb = make_batches(tok, hyps, refs, a.host_batch)[0]
    torch.set_num_threads(os.cpu_count() or 1)
    ref = bo.make_model(cfg, seed=5, perturb=False)
    t0 = time.perf_counter()
    bto.step(ref, hb["input_ids"], hb["attention_mask"], hb["labels"])
    res["host_fp32_step"] = dict(sents=a.host_batch, seconds=time.perf_counter() - t0, threads=torch.get_num_threads())
    print(json.dumps(res["host_fp32_step"]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
