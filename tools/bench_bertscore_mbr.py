"""BERTScore MBR (RMBR) throughput on one B200: the embedding pass (pllb_embed) and the pair kernel
(pllb_bertscore) timed separately with device events, then hypotheses/s end to end from strings
(RMBR.utility_functions.BertScoreFunction.pairwise: tokenisation, deduplication, embedding, pair
recall, copies back).  Not bench.py's workload; one JSON line on stdout (and in --out if given).

    python tools/bench_bertscore_mbr.py [--utts 7176] [--layers 8] [--reps 5] [--cpu-utts 3] [--out FILE]

Workload: C2 shape — synthetic AISHELL-1-test-shaped 10-best lists (synth.make_nbest, 7 176 utterances,
seed 0), bert-base-chinese shape with random init (seed 10), encoder truncated to 8 layers (bert_score's
choice for bert-base-chinese), bf16 operands; every ordered pair (i, j != i) of every utterance, grouped
by candidate as mbr_decode emits them.  Each timed stage is warmed up once and moves far more than the
126 MB of L2 (3.7 GB of fp32 states).  Bounds: the embedding pass against the data-sheet dense bf16
rate (2 250 TFLOP/s); the pair kernel against the fp32 SIMT rate computed from the card's SM count and
maximum SM clock read in the same run (128 FMA lanes per SM) and against HBM bandwidth (7.7 TB/s) for
one read of the states.  CPU arm: oracle/bertscore_oracle.py (transformers.BertModel + bert_score's
matching restated in torch fp32, all host threads) on the first --cpu-utts utterances, labelled "port":
bert_score itself is not installed.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BF16_PEAK = 2250e12
HBM_BW = 7.7e12


def _smi(fields):
    out = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True).stdout.strip().split("\n")[0]
    return [x.strip() for x in out.split(",")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=7176)
    ap.add_argument("--layers", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu-utts", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.utts < 1 or args.reps < 1 or args.cpu_utts < 0:
        ap.error("--utts and --reps must be >= 1, --cpu-utts >= 0")
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import torch
    from asr_rescoring_b200 import engine, synth
    from asr_rescoring_b200.RMBR.utility_functions import BertScoreFunction
    from asr_rescoring_b200.tokenizer import SyntheticCharTokenizer

    n = 10
    cfg = synth.BERT_BASE_CHINESE
    H, I, NL = cfg["hidden"], cfg["intermediate"], args.layers
    sd = synth.random_init_state_dict(cfg, 10)
    nb = synth.make_nbest(args.utts, n, seed=0)
    tok, off = nb.packed_tokens()
    L = np.diff(off)
    T = L + 2
    rows = int(T.sum())
    row_off = np.zeros(len(T) + 1, np.int64)
    np.cumsum(T, out=row_off[1:])
    ii, jj = np.nonzero(~np.eye(n, dtype=bool))
    base = (np.arange(args.utts) * n)[:, None]
    cand = (base + ii[None]).reshape(-1).astype(np.int32)
    ref = (base + jj[None]).reshape(-1).astype(np.int32)
    # shape arithmetic
    emb_flops = float(NL * (T * (8 * H * H + 4 * H * I) + 4 * T * T * H).sum())
    pair_flops = float((2.0 * H * T[cand] * (T[ref] - 2)).sum() + 2.0 * H * rows)
    state_bytes = 4.0 * rows * H
    name = torch.cuda.get_device_name(0)
    power_limit, sms_clock = _smi("power.limit,clocks.max.sm")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    fp32_peak = sms * 128 * 2 * float(sms_clock) * 1e6

    def timed(fn, reps):
        fn()                                           # warm-up
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            out = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / 1e3 / reps, out

    with engine.PllScorer(sd, cfg, operand_dtype="bf16") as sc:
        t = torch.from_numpy(tok).cuda()
        buf = torch.empty(rows, H, dtype=torch.float32, device="cuda")
        s_emb, emb = timed(lambda: sc.embed(t, off, NL, out=buf), args.reps)
        out = torch.empty(len(cand), dtype=torch.float32, device="cuda")
        s_pair, rec = timed(lambda: sc.bertscore(emb, row_off, cand, ref, out=out), args.reps)
        recall_mean = float(rec.mean())
        del buf, emb, t
    torch.cuda.empty_cache()
    util = BertScoreFunction(sd, SyntheticCharTokenizer(), num_layers=NL, cfg=cfg, operand_dtype="bf16")
    util.pairwise(nb.hyps[:50], n)                    # warm-up (tokenizer table, allocations)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    U = util.pairwise(nb.hyps, n)
    e2e = time.perf_counter() - t0
    util.close()
    cpu = None
    if args.cpu_utts > 0:
        import bench
        from oracle import bertscore_oracle as bo
        torch.set_num_threads(bench.host_threads())
        tk = SyntheticCharTokenizer()
        o = bo.OracleBertScore(sd, cfg, tk.encode, NL)
        sub = nb.hyps[:args.cpu_utts]
        t0 = time.perf_counter()
        bo.mbr_decode(n, sub, o)
        cdt = time.perf_counter() - t0
        cpu = dict(kind="port", hyps_per_s=n * len(sub) / cdt, seconds=cdt, cores=torch.get_num_threads(),
                   sample=f"{len(sub)} utterances x {n}-best through oracle/bertscore_oracle.py mbr_decode "
                          "(transformers.BertModel fp32 + bert_score's matching, one pair per batch)")
    res = {"metric": "BERTScore MBR hypotheses/sec end to end from strings", "unit": "hyps/s",
           "value": len(L) / e2e, "device": name, "power_limit_w": float(power_limit),
           "max_sm_clock_mhz": float(sms_clock),
           "config": {"workload": f"C2 shape: {args.utts} utterances x {n}-best, bert-base-chinese shape, random init, "
                                  f"{NL} layers, bf16 operands, every ordered pair", "reps": args.reps},
           "shape": {"hyps": int(len(L)), "rows": rows, "mean_T": float(T.mean()), "pairs": int(len(cand)),
                     "embed_flops": emb_flops, "pair_flops": pair_flops, "state_bytes": state_bytes},
           "embed": {"seconds": s_emb, "tflops_per_s": emb_flops / s_emb / 1e12,
                     "share_of_bf16_bound": emb_flops / BF16_PEAK / s_emb},
           "pair_kernel": {"seconds": s_pair, "tflops_per_s": pair_flops / s_pair / 1e12,
                           "fp32_simt_peak_tflops": fp32_peak / 1e12,
                           "share_of_fp32_bound": pair_flops / fp32_peak / s_pair,
                           "share_of_hbm_bound": state_bytes / HBM_BW / s_pair, "mean_recall": recall_mean},
           "end_to_end": {"seconds": e2e, "hyps_per_s": len(L) / e2e, "mean_offdiag_recall":
                          float(U[:, ~np.eye(n, dtype=bool)].mean())},
           "cpu_baseline": cpu, "ratio": (len(L) / e2e) / cpu["hyps_per_s"] if cpu else None}
    os.dup2(real_stdout, 1)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
