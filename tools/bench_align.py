"""Edit-operation alignment throughput on one B200 (pllb_align, DESIGN.md §3.10).  Not bench.py's
workload; one JSON line on stdout (and in --out if given).

    python tools/bench_align.py [--utts 7176] [--long-pairs 2000] [--reps 20] [--cpu-long-pairs 100] [--out FILE]

Workloads: the C2 shape (synth.make_nbest(7176, 10, seed 0): 71 760 (ref, hyp) pairs of stripped
code points, about 15 x 15 cells each; every pair keeps its backtrace codes in shared memory) and a
long-pair shape (--long-pairs pairs, both sides 512-1 024 symbols, the hypothesis a 10 %-edited copy
of the reference, seed 1; codes in the global scratch region).  Device arms, timed with CUDA events
over --reps launches after one warm-up launch, inputs resident on the device: pllb_align and
pllb_levenshtein on the same pairs (the backtrace's cost on top of the distance).  End to end:
cer_clients.hyp_alignment from the {utt: {hyp_k: text}} dicts (strip, packing, copies, kernel,
building the lists), host clock.  CPU arm: the C restatement oracle/align_oracle.c on one host thread,
labelled "port" (the reference's align.py is pure Python and not installed here); for the long
shape on the first --cpu-long-pairs pairs.  The pair stage is latency-bound (a few hundred cells
per warp), so no share of a peak is claimed.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _smi(fields):
    out = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True).stdout.strip().split("\n")[0]
    return [x.strip() for x in out.split(",")]


def _long_pairs(n, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    refs, hyps = [], []
    for _ in range(n):
        r = rng.integers(0, 4000, size=int(rng.integers(512, 1025))).astype(np.int32)
        h = r.copy()
        m = rng.random(len(h)) < 0.1
        h[m] = rng.integers(0, 4000, size=int(m.sum()))
        lb = int(rng.integers(512, 1025))
        h = np.concatenate([h, rng.integers(0, 4000, size=max(lb - len(h), 0)).astype(np.int32)])[:lb]
        refs.append(r)
        hyps.append(h)
    off = lambda xs: np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.int64)
    return np.concatenate(refs), off(refs), np.concatenate(hyps), off(hyps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=7176)
    ap.add_argument("--long-pairs", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cpu-long-pairs", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.utts < 1 or args.long_pairs < 1 or args.reps < 1 or args.cpu_long_pairs < 0:
        ap.error("--utts, --long-pairs and --reps must be >= 1, --cpu-long-pairs >= 0")
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import torch
    from oracle import align_oracle
    from asr_rescoring_b200 import _lib, cer_clients, engine, synth

    lib = _lib.load()
    _lib.require_device()
    name = torch.cuda.get_device_name(0)
    power_limit, sm_clock = _smi("power.limit,clocks.max.sm")
    stream = torch.cuda.current_stream().cuda_stream

    def device_arms(rc, ro, hc, ho, pair_ref):
        n = len(pair_ref)
        max_len = int(max(np.diff(ro).max(initial=0), np.diff(ho).max(initial=0)))
        ops_off = np.zeros(n + 1, np.int64)
        np.cumsum(np.diff(ro)[pair_ref] + np.diff(ho), out=ops_off[1:])
        d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (rc, ro, hc, ho, pair_ref, ops_off)]
        ops = torch.empty(max(int(ops_off[-1]), 1), dtype=torch.uint8, device="cuda")
        n_ops = torch.empty(n, dtype=torch.int32, device="cuda")
        counts = torch.empty((n, 4), dtype=torch.int32, device="cuda")
        dist = torch.empty(n, dtype=torch.int32, device="cuda")
        p = [x.data_ptr() for x in d]
        align = lambda: _lib.check(lib.pllb_align(p[0], p[1], p[2], p[3], p[4], n, max_len, p[5], ops.data_ptr(),
                                                  n_ops.data_ptr(), counts.data_ptr(), stream))
        lev = lambda: _lib.check(lib.pllb_levenshtein(p[0], p[1], p[2], p[3], p[4], n, max_len, dist.data_ptr(), stream))

        def timed(fn):
            fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / 1e3 / args.reps

        t_align, t_lev = timed(align), timed(lev)
        # alternate once more so a drifting clock shows up as a spread
        t_align2, t_lev2 = timed(align), timed(lev)
        edits = counts[:, 1:].sum(dim=1)
        assert torch.equal(edits, dist), "align S+I+D differs from the Levenshtein distance"
        cells = float((np.diff(ro)[pair_ref] * np.diff(ho)).sum())
        return {"pairs": n, "cells": cells, "max_len": max_len,
                "align_seconds": [t_align, t_align2], "levenshtein_seconds": [t_lev, t_lev2],
                "align_over_levenshtein": min(t_align, t_align2) / min(t_lev, t_lev2),
                "align_pairs_per_s": n / min(t_align, t_align2), "align_gcells_per_s": cells / min(t_align, t_align2) / 1e9,
                "edits": int(edits.sum())}

    def port(rc, ro, hc, ho, pair_ref):
        t0 = time.perf_counter()
        align_oracle.align_batch(rc, ro, hc, ho, pair_ref)
        dt = time.perf_counter() - t0
        return {"kind": "port", "what": "oracle/align_oracle.c full-table backtrace, 1 host thread", "pairs": len(pair_ref),
                "seconds": dt, "pairs_per_s": len(pair_ref) / dt}

    nb = synth.make_nbest(args.utts, 10, seed=0)
    refs = [r.strip() for r in nb.refs]
    hyps = [h.strip() for hs in nb.hyps for h in hs]
    rc, ro = engine.pack_strings(refs)
    hc, ho = engine.pack_strings(hyps)
    pr = np.repeat(np.arange(len(refs), dtype=np.int32), 10)
    c2 = device_arms(rc, ro, hc, ho, pr)
    c2["port"] = port(rc, ro, hc, ho, pr)
    c2["port"]["ratio_align_kernel"] = c2["align_pairs_per_s"] / c2["port"]["pairs_per_s"]
    ht, rt = nb.hyps_text(), nb.ref_text()
    cer_clients.hyp_alignment(dict(list(ht.items())[:100]), rt)       # warm-up
    e2e = []
    for _ in range(3):
        t0 = time.perf_counter()
        cer_clients.hyp_alignment(ht, rt)
        e2e.append(time.perf_counter() - t0)
    c2["hyp_alignment_end_to_end"] = {"seconds": e2e, "pairs_per_s": len(hyps) / min(e2e),
                                      "port_ratio": (len(hyps) / min(e2e)) / c2["port"]["pairs_per_s"]}

    lrc, lro, lhc, lho = _long_pairs(args.long_pairs, 1)
    lpr = np.arange(args.long_pairs, dtype=np.int32)
    lg = device_arms(lrc, lro, lhc, lho, lpr)
    if args.cpu_long_pairs > 0:
        k = min(args.cpu_long_pairs, args.long_pairs)
        lg["port"] = port(lrc, lro[:k + 1], lhc, lho[:k + 1], lpr[:k])
        lg["port"]["ratio_align_kernel"] = lg["align_pairs_per_s"] / lg["port"]["pairs_per_s"]

    res = {"metric": "edit-operation alignment pairs/sec, C2 shape, pllb_align kernel", "unit": "pairs/s",
           "value": c2["align_pairs_per_s"], "device": name, "power_limit_w": float(power_limit),
           "max_sm_clock_mhz": float(sm_clock), "reps": args.reps,
           "c2": dict(c2, workload=f"synth.make_nbest({args.utts}, 10, seed 0), stripped code points"),
           "long": dict(lg, workload=f"{args.long_pairs} pairs, 512-1024 symbols per side, 10 % edits, seed 1")}
    os.dup2(real_stdout, 1)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
