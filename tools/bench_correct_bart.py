"""CorrectBart one_hyp generation throughput on the device (DESIGN.md §3.11).

C2 1-best (synth.make_nbest(7176, 10), hyp_1), bart-base-chinese shape (6 + 6 layers, d_model 768,
FFN 3072, vocab 21128), random init, max_length 50, both operand types.  Warm-up pass, then CUDA-event
timed passes (pllb_s2s timing: encoder, cross K/V, decoder layers, LM head + argmax).  Next to it: the
fp32 oracle's generate() on all host threads over a small sample.  Writes profiles/correct_bart_bench.json
(or --out).

--num-beams K > 1 measures beam search instead (DESIGN.md §3.12) and writes
profiles/correct_bart_beam_bench.json: per operand type, greedy and K beams at the default max_rows, K
beams in one chunk (max_rows = K * utts), and K beams with an EOS bias on final_logits_bias (--eos-bias),
meant to let early stopping end the run before max_length - 1 steps; the JSON records the steps run.  All in one process, next to the GPU's name and
power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_context():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=7176)
    ap.add_argument("--max-length", type=int, default=50)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--oracle-sample", type=int, default=16)
    ap.add_argument("--out", default=None)
    ap.add_argument("--num-beams", type=int, default=1)
    ap.add_argument("--eos-bias", type=float, default=4.0, help="beam runs: bias added to EOS in the EOS-bias run")
    a = ap.parse_args()
    if a.num_beams > 1:
        return bench_beam(a)
    a.out = a.out or os.path.join(ROOT, "profiles", "correct_bart_bench.json")
    import torch
    from asr_rescoring_b200 import engine, synth
    from oracle import bart_oracle as bo

    cfg = bo.bart_config(d_model=768, layers=6, ffn=3072, vocab=21128, max_position=512)
    m = bo.make_model(cfg, seed=5)
    nb = synth.make_nbest(a.utts, 10)
    sents = [[synth.synthetic_token_id(c) for c in hs[0]] for hs in nb.hyps]
    off = np.zeros(len(sents) + 1, np.int64)
    np.cumsum([len(s) for s in sents], out=off[1:])
    tok = np.array([t for s in sents for t in s], np.int32)
    gen = engine.generation_settings(cfg.to_dict(), max_length=a.max_length, decoder_start_token_id=2,
                                     eos_token_id=102, pad_token_id=0)
    H, I, V, NL = 768, 3072, 21128, 6
    res = dict(workload=dict(utts=a.utts, input_tokens=int(off[-1]), max_length=a.max_length, shape="6+6 x 768, FFN 3072, V 21128",
                             init="random (oracle make_model, seed 5)"), gpu=gpu_context(), modes={})
    for dtype in ("bf16", "fp16"):
        with engine.Seq2SeqGenerator(m.state_dict(), cfg.to_dict(), device=0, operand_dtype=dtype) as g:
            g.generate_packed(tok, off, gen)                         # warm-up: every shape of the timed passes
            g.set_timing(True)
            runs = []
            for _ in range(a.passes):
                g.reset_stats()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ids, lens = g.generate_packed(tok, off, gen)
                wall = time.perf_counter() - t0
                st = g.stats()
                runs.append((wall, st))
            wall = float(np.median([r[0] for r in runs]))
            st = sorted(runs, key=lambda r: r[0])[len(runs) // 2][1]
            gen_tokens = int((lens - 1).sum())
            dev_s = st["total_ms"] / 1e3
            res["modes"][dtype] = dict(
                wall_s=wall, device_s=dev_s, sentences_per_s=a.utts / wall, generated_tokens_per_s=gen_tokens / wall,
                generated_tokens=gen_tokens, mean_generated_length=float((lens - 1).mean()),
                sentences_with_eos=int((ids[np.arange(len(lens)), lens - 1] == 102).sum()),
                steps=int(st["steps"]), chunks=int(st["chunks"]),
                launches_per_step=st["kernel_launches"] / max(st["steps"], 1),
                split_ms=dict(encoder=st["enc_ms"], cross_kv=st["cross_kv_ms"], decoder_layers=st["dec_layers_ms"],
                              lm_head_argmax=st["head_ms"]),
                gemm_tflop=st["gemm_flops"] / 1e12, algorithmic_tflops_per_s=st["gemm_flops"] / 1e12 / dev_s,
                workspace_gb=st["workspace_bytes"] / 1e9, wall_s_all_passes=[r[0] for r in runs])
            print(dtype, json.dumps(res["modes"][dtype]), flush=True)
    # the oracle's generate() on all host threads over a small sample, for the ratio
    torch.set_num_threads(os.cpu_count() or 1)
    sample = sents[:a.oracle_sample]
    t0 = time.perf_counter()
    bo.hf_generate(m, sample, 101, 102, gen)
    t = time.perf_counter() - t0
    res["oracle_cpu"] = dict(sentences=len(sample), threads=torch.get_num_threads(), seconds=t,
                             sentences_per_s=len(sample) / t)
    res["speedup_vs_oracle_cpu"] = {k: v["sentences_per_s"] / res["oracle_cpu"]["sentences_per_s"]
                                    for k, v in res["modes"].items()}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


def timed(g, tok, off, settings, passes, beam):
    """Warm-up, then `passes` timed calls; the median pass's wall time and stats and the last result."""
    import torch
    run = (lambda: g.beam_search_packed(tok, off, settings)) if beam else (lambda: g.generate_packed(tok, off, settings))
    run()
    g.set_timing(True)
    runs = []
    for _ in range(passes):
        g.reset_stats()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = run()
        runs.append((time.perf_counter() - t0, g.stats()))
    g.set_timing(False)
    wall = float(np.median([r[0] for r in runs]))
    st = sorted(runs, key=lambda r: r[0])[len(runs) // 2][1]
    lens = out[1][:, 0] if beam else out[1]
    ids = out[0][:, 0] if beam else out[0]
    gen_tokens = int((lens - 1).sum())
    dev_s = st["total_ms"] / 1e3
    return dict(
        wall_s=wall, device_s=dev_s, sentences_per_s=len(lens) / wall, generated_tokens_per_s=gen_tokens / wall,
        generated_tokens=gen_tokens, mean_generated_length=float((lens - 1).mean()),
        sentences_with_eos=int((ids[np.arange(len(lens)), lens - 1] == 102).sum()),
        steps=int(st["steps"]), chunks=int(st["chunks"]), launches_per_step=st["kernel_launches"] / max(st["steps"], 1),
        split_ms=dict(encoder=st["enc_ms"], cross_kv=st["cross_kv_ms"], decoder_layers=st["dec_layers_ms"],
                      lm_head_and_selection=st["head_ms"]),
        gemm_tflop=st["gemm_flops"] / 1e12, algorithmic_tflops_per_s=st["gemm_flops"] / 1e12 / dev_s,
        workspace_gb=st["workspace_bytes"] / 1e9, wall_s_all_passes=[r[0] for r in runs])


def bench_beam(a):
    import torch
    from asr_rescoring_b200 import engine, synth
    from oracle import bart_oracle as bo

    out = a.out or os.path.join(ROOT, "profiles", "correct_bart_beam_bench.json")
    cfg = bo.bart_config(d_model=768, layers=6, ffn=3072, vocab=21128, max_position=512)
    m = bo.make_model(cfg, seed=5)
    nb = synth.make_nbest(a.utts, 10)
    sents = [[synth.synthetic_token_id(c) for c in hs[0]] for hs in nb.hyps]
    off = np.zeros(len(sents) + 1, np.int64)
    np.cumsum([len(s) for s in sents], out=off[1:])
    tok = np.array([t for s in sents for t in s], np.int32)
    base = dict(max_length=a.max_length, decoder_start_token_id=2, eos_token_id=102, pad_token_id=0)
    greedy = engine.generation_settings(cfg.to_dict(), **base)
    beam = engine.beam_settings(cfg.to_dict(), num_beams=a.num_beams, **base)
    one_chunk = a.num_beams * a.utts
    res = dict(workload=dict(utts=a.utts, input_tokens=int(off[-1]), max_length=a.max_length, num_beams=a.num_beams,
                             length_penalty=beam["length_penalty"], early_stopping=beam["early_stopping"],
                             shape="6+6 x 768, FFN 3072, V 21128", init="random (oracle make_model, seed 5)",
                             eos_bias=a.eos_bias),
               gpu=gpu_context(), modes={})
    sd = m.state_dict()
    sd_eos = dict(sd)
    sd_eos["final_logits_bias"] = sd["final_logits_bias"].clone()
    sd_eos["final_logits_bias"][0, 102] += a.eos_bias
    for dtype in ("bf16", "fp16"):
        runs = (("greedy", sd, 0, greedy, False), (f"beam{a.num_beams}", sd, 0, beam, True),
                (f"beam{a.num_beams}_one_chunk", sd, one_chunk, beam, True),
                (f"beam{a.num_beams}_eos_bias", sd_eos, 0, beam, True))
        for name, weights, max_rows, settings, is_beam in runs:
            with engine.Seq2SeqGenerator(weights, cfg.to_dict(), device=0, operand_dtype=dtype, max_rows=max_rows) as g:
                r = timed(g, tok, off, settings, a.passes, is_beam)
            r["max_rows"] = max_rows or 8192
            res["modes"][f"{dtype}_{name}"] = r
            print(dtype, name, json.dumps(r), flush=True)
        g_s = res["modes"][f"{dtype}_greedy"]["wall_s"]
        res["modes"][f"{dtype}_beam{a.num_beams}"]["cost_vs_greedy"] = res["modes"][f"{dtype}_beam{a.num_beams}"]["wall_s"] / g_s
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
