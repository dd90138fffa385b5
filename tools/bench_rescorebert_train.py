"""RescoreBert distillation throughput: hypotheses per second of a training step (engine.ClsTrainer,
pllb_cls_train_*) on one B200 next to the autograd restatement on the host cores.  Not bench.py's
workload; one JSON line on stdout.

    python tools/bench_rescorebert_train.py [--utts 4,32] [--batches 8] [--warmup 2] [--passes 10] [--layers 12] [--cpu-batches 1]

Workload: bert-base-chinese shape, random init (seed 10), dropout 0.1, AdamW lr 1e-5, MD + MWER (weights 1,
am_weight 1).  Synthetic AISHELL-1-test-shaped 10-best lists (synth.make_nbest): AM scores from the list,
CER = applied edits / reference length, teacher PLL = synth.synthetic_lm_scores (the step's cost does not
depend on the values).  For each batch size (utterances per batch, 10 hypotheses each) `--batches` distinct
padded batches; `--warmup` untimed passes over them (a batch shape runs eagerly once and is captured as a
CUDA graph the second time), then `--passes` timed passes — the steady state of every epoch after the second.
One host sync per step (the loss and the scores come back).  CPU arm: oracle/rescorebert_train_oracle.py
(plain torch fp32, all host threads) for `--cpu-batches` batches of the smallest size, labelled "port":
the reference's training loop is not installed.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", default="4,32", help="utterances per batch, comma-separated")
    ap.add_argument("--batches", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--layers", type=int, default=12)
    ap.add_argument("--cpu-batches", type=int, default=1)
    args = ap.parse_args()
    if args.batches < 1 or args.warmup < 0 or args.passes < 1:
        ap.error("--batches and --passes must be >= 1, --warmup >= 0")
    sizes = [int(x) for x in args.utts.split(",")]
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import bench
    from asr_rescoring_b200 import engine, synth
    from asr_rescoring_b200.RescoreBert import train as rb_train

    cfg = dict(synth.BERT_BASE_CHINESE, num_layers=args.layers)
    sd = synth.random_rescorebert_state_dict(cfg, 10)
    nb = synth.make_nbest(max(sizes) * args.batches, 10, seed=0)
    tok, off = nb.packed_tokens()
    lm = synth.synthetic_lm_scores(nb)
    tokens, pll, am, cer = {}, {}, {}, {}
    for u, utt in enumerate(nb.utt_ids):
        keys = [f"hyp_{k + 1}" for k in range(10)]
        tokens[utt] = {h: [int(t) for t in tok[off[u * 10 + k]:off[u * 10 + k + 1]]] for k, h in enumerate(keys)}
        pll[utt] = {h: float(lm[u, k]) for k, h in enumerate(keys)}
        am[utt] = {h: float(nb.am[u, k]) for k, h in enumerate(keys)}
        cer[utt] = {h: float(nb.edits[u, k]) / len(nb.refs[u]) for k, h in enumerate(keys)}
    weights = dict(md_weight=1.0, mwer_weight=1.0, am_weight=1.0)
    gpu = {}
    clocks = None
    for n_utt in sizes:
        batches = rb_train.make_batches(tokens, pll, am, cer, n_utt)[:args.batches]
        rows, seq = rb_train.batch_capacity(batches)
        with engine.ClsTrainer(sd, cfg, lr=1e-5, hidden_dropout=0.1, attention_dropout=0.1, seed=10, max_rows=rows,
                               max_seq=seq, **weights) as tr:
            tr.reset_optimizer(1e-5)
            for _ in range(args.warmup):
                rb_train.run_one_epoch(tr, batches, True)
            l0, r0 = tr.kernel_launches(), tr.graph_replays()
            sampler = bench.ClockSampler(torch.cuda.current_device())
            sampler.start()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loss = [rb_train.run_one_epoch(tr, batches, True) for _ in range(args.passes)][-1]
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            clocks = sampler.stop()
            steps = args.passes * len(batches)
            hyps = args.passes * sum(b["input_ids"].shape[0] for b in batches)
            gpu[f"{n_utt}_utts"] = dict(
                hyps_per_s=hyps / dt, ms_per_step=1e3 * dt / steps, hyps_per_step=hyps / steps, timed_seconds=dt,
                padded_rows_per_step=sum(b["input_ids"].size for b in batches) / len(batches),
                launches_per_step=(tr.kernel_launches() - l0) / steps,
                graph_replays_in_timed_steps=f"{tr.graph_replays() - r0} of {steps}",
                distinct_batch_shapes=len({b["input_ids"].shape for b in batches}), last_pass_mean_loss=loss,
                workspace_gb=tr.workspace_bytes() / 1e9, clocks=clocks)
    cpu = None
    if args.cpu_batches > 0:
        from oracle import rescorebert_train_oracle as rto
        threads = bench.host_threads()
        torch.set_num_threads(threads)
        sample = rb_train.make_batches(tokens, pll, am, cer, min(sizes))[:args.cpu_batches]
        params = rto.parameters(sd)
        t0 = time.perf_counter()
        rto.run_steps(params, cfg, sample, 1e-5, **weights)
        cdt = time.perf_counter() - t0
        hyps = sum(b["input_ids"].shape[0] for b in sample)
        cpu = dict(hyps_per_s=hyps / cdt, seconds=cdt, cores=threads, kind="port",
                   sample=f"{len(sample)} batches of {min(sizes)} utterances through oracle/rescorebert_train_oracle.py "
                          "(torch fp32 autograd + torch.optim.AdamW, dropout 0)")
    os.dup2(real_stdout, 1)
    first = f"{sizes[0]}_utts"
    print(json.dumps({"metric": "RescoreBert distillation hypotheses/sec", "unit": "hyps/s", "value": gpu[first]["hyps_per_s"],
                      "device": torch.cuda.get_device_name(0), "power_limit_w": (clocks or {}).get("power_limit_w"),
                      "config": {"workload": f"bert-base-chinese shape, {cfg['num_layers']} layers, random init, AISHELL-1-shaped "
                                             "10-best lists, dropout 0.1, AdamW lr 1e-5, MD + MWER",
                                 "batches": args.batches, "warmup_passes": args.warmup, "timed_passes": args.passes,
                                 "utts_per_batch": sizes},
                      "dtype": "bf16 operands, fp32 master weights / gradients / moments", "gpu": gpu, "cpu_baseline": cpu,
                      "ratio": gpu[first]["hyps_per_s"] / cpu["hyps_per_s"] if cpu else None}), flush=True)


if __name__ == "__main__":
    main()
