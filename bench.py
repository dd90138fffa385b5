"""bench.py — N-best PLL hypotheses/sec of the MLM-PLL scoring path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c1|c2|c4|c5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A step is one pass of the whole hot path over the workload: stages 1-3 (on-device masked-copy
expansion, BERT encoder, masked-row MLM head -> per-hypothesis PLL) and stage 4 (all (ref, hyp)
Levenshtein distances + 101-point weight sweep with per-utterance argmax).

Workloads (BASELINE.json configs; synthetic data from synth.py, random-init weights, seed 10):
  c2 (default)  7 176 AISHELL-1-test-shaped utterances x 10-best, bert-base-chinese  (configs[1]; with
                --gpus N > 1 the SAME list sharded by utterance = configs[2], "scaling": "strong")
  c1            the first 100 utterances of c2                                         (configs[0])
  c4            50-best, length 8..64, bert-large-shaped 24L/1024H, fp16 operands      (configs[3])
  c5            combiner only: 7 176 x 50-best, 101 weights, Levenshtein + sweep        (configs[4])

N > 1 (strong scaling, the default): one utterance list, LPT-partitioned over the ranks by
expanded-token cost; every step ends with the two collectives of the path INSIDE the timed
region — an NCCL all_gather of the per-hypothesis scores and an all_reduce of the per-weight
edit sums + reference length.  `--scaling weak` keeps round 1's independent replicas.

value   : device-resident inputs, whole job, max over ranks, CUDA-event timed (no per-launch
          events inside this region; the per-kind GEMM breakdown comes from one extra step).
e2e     : the same through the host-buffer C-ABI calls (pllb_score_host, pllb_levenshtein_host,
          pllb_rescore_sweep_host; c5: the drop-in rescore.find_best_weight): H2D and D2H inside.
roofline: the dominant kernel of the step (largest summed launch time of the per-kind
          breakdown): executed FLOPs (sum of 2*M*N*K over its launches) / summed launch durations
          from CUDA events recorded on the launch stream; `by_kind` carries every GEMM kind and
          `gemm_family` the round-1 aggregate.  `traffic` is a profile constant (ncu --set full of
          the same kernel, profiles/roofline_traffic.json), not measured by this run.
cpu_baseline / --impl reference: the reference's own CPU code from baseline/_ref (unmodified
          MLM_PLL/main.py set_dataloader + run_one_epoch on transformers.BertForMaskedLM; c5:
          rescore.find_best_weight under the jiwer stand-in), all host threads, bounded sample;
          falls back to the oracle port (kind "port") only when baseline/_ref is absent.
stdout  : exactly one JSON line (library banners are redirected to stderr).
--dump-outputs DIR: after the timed steps, what the last timed step computed, as rank 0's caller
          receives it, goes to DIR/<name>.npy: pll (per-hypothesis PLL, float64; N > 1 strong: every
          hypothesis in global order after the gather; not for c5, where it is an input), distance
          (per-hypothesis Levenshtein distance, float32), argmax ([weight, utterance] index of the
          chosen hypothesis, float32), edit_sums (per-weight edit sum, float64; N > 1 strong: after the
          all_reduce).  Inputs are seeded, so two builds run with the same arguments can be compared
          file by file.  Over 64 MB in all, an array keeps a fixed, seeded sample of its last axis
          (positions in <name>_index.npy).
"""
from __future__ import annotations

import argparse
import ctypes
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "N-best PLL hypotheses/sec"
UNIT = "hyps/s"

WORKLOADS = {
    "c1": dict(n_utts=100, n_best=10, model="bert-base-chinese", min_len=None, max_len=None, dtype="bf16+fp16head",
               desc="c1: 100 synthetic AISHELL-1-shaped utterances x 10-best, random-init bert-base-chinese, "
                    "PLL + 101-point weight sweep"),
    "c2": dict(n_utts=7176, n_best=10, model="bert-base-chinese", min_len=None, max_len=None, dtype="bf16+fp16head",
               desc="c2: AISHELL-1-test-shaped 7176 utterances x 10-best, random-init bert-base-chinese, "
                    "PLL + 101-point weight sweep"),
    # fp16 operands are part of this workload's definition, not a silent switch: with bf16 the
    # 24-layer encoder at L <= 64 misses the 0.05-nat bound (tests/test_gpu_parity.py::
    # test_config4_24_layers_L64_vs_reference_golden measures both); same tensor-core rate.
    "c4": dict(n_utts=7176, n_best=50, model="bert-large-shaped", min_len=8, max_len=64, dtype="fp16", sample_utts=150,
               desc="c4: 7176 utterances x 50-best, length 8..64, bert-large-shaped encoder (24L/1024H), "
                    "PLL + 101-point weight sweep"),
    "c5": dict(n_utts=7176, n_best=50, model=None, min_len=None, max_len=None, dtype="f64",
               desc="c5: combiner only, 7176 utterances x 50-best, AM + PLL weight grid (101 points) argmax + "
                    "Levenshtein CER over the full test set"),
}
KIND_KERNEL = {
    "qkv": "gemm_tcgen05_kernel<EPI_BIAS_BF16, cta_group::2>", "attn_out": "gemm_ln_kernel<H/256, staged>",
    "ffn1": "gemm_tcgen05_kernel<EPI_BIAS_GELU_BF16, W multicast>", "ffn2": "gemm_ln_kernel<H/256, direct>",
    "head_transform": "gemm_tcgen05_kernel<EPI_BIAS_GELU_F32>", "decoder_lse": "gemm_tcgen05_kernel<EPI_LSE>",
}


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--utts", type=int, default=0, help="override the number of utterances")
    ap.add_argument("--chunk-tokens", type=int, default=1 << 20)
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="N > 1: strong (default; one list sharded over the ranks) or weak (a full list per rank)")
    ap.add_argument("--cpu-sample-hyps", type=int, default=0, help="hypotheses in the bounded CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--operand-dtype", default=None,
                    help="GEMM operand type; default = the workload's (bf16 encoder + fp16 MLM head; fp16 for c4), always "
                         "reported in `dtype`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the timed path of --impl b200")
    return args


def model_cfg(name):
    from asr_rescoring_b200 import synth
    return {"bert-base-chinese": synth.BERT_BASE_CHINESE, "bert-large-shaped": synth.BERT_LARGE_SHAPED}[name]


def gemm_flops(lengths, cfg):
    """Algorithmic FLOPs of the dense GEMMs (SURVEY.md §8d): per hypothesis of L tokens,
    T = L+2: L*[T*NL*(8H^2+4HI) + 2H^2 + 2HV]."""
    H, I, NL, V = cfg["hidden"], cfg["intermediate"], cfg["num_layers"], cfg["vocab"]
    L = np.asarray(lengths, np.float64)
    return float((L * ((L + 2) * NL * (8 * H * H + 4 * H * I) + 2 * H * H + 2 * H * V)).sum())


def total_flops(lengths, cfg):
    H, NL = cfg["hidden"], cfg["num_layers"]
    L = np.asarray(lengths, np.float64)
    return gemm_flops(lengths, cfg) + float((L * NL * 4 * (L + 2) ** 2 * H).sum())


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,power.limit")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self._halt = threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})

        def _num(col):
            vals = []
            for smp in self.samples:
                try:
                    vals.append(float(smp[col]))
                except (IndexError, ValueError):
                    pass
            return float(np.median(vals)) if vals else None

        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples), "power_w": _num(6), "power_limit_w": _num(7)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["bf16_tflops_sustained"]), float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json: bf16_tflops_sustained, hbm_gbs)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained bf16, ~6.65 TB/s copy)"


def host_threads() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


# ------------------------------------------------------------------------------------ CPU arms
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
SHIMS = os.path.join(ROOT, "baseline", "shims")


def _load_reference_module(name: str, rel: str, cwd_rel: str):
    """Import an UNMODIFIED reference file from baseline/_ref by path (ruamel.yaml / jiwer come from
    baseline/shims).  Returns None when the install is absent."""
    path = os.path.join(REF_DIR, rel)
    if not os.path.exists(path):
        return None
    for p in (SHIMS, os.path.join(REF_DIR, cwd_rel)):
        if p not in sys.path:
            sys.path.insert(0, p)
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    cwd = os.getcwd()
    os.chdir(os.path.join(REF_DIR, cwd_rel))         # MLM_PLL/main.py does sys.path.append("..")
    try:
        spec.loader.exec_module(mod)
    finally:
        os.chdir(cwd)
    return mod


class CpuPllArm:
    """The reference's torch CPU scoring path on the first n hypotheses of a workload."""

    def __init__(self, cfg, sd):
        import torch
        self.cfg, self.sd = cfg, sd
        self.threads = host_threads()
        torch.set_num_threads(self.threads)          # torchrun exports OMP_NUM_THREADS=1
        self.ref_main = _load_reference_module("ref_mlm_pll_main", os.path.join("MLM_PLL", "main.py"), "MLM_PLL")
        self.kind = "reference" if self.ref_main is not None else "port"
        self.model = None
        if self.ref_main is not None:
            from transformers import BertConfig, BertForMaskedLM
            hf = BertForMaskedLM(BertConfig(
                vocab_size=cfg["vocab"], hidden_size=cfg["hidden"], num_hidden_layers=cfg["num_layers"],
                num_attention_heads=cfg["num_heads"], intermediate_size=cfg["intermediate"],
                max_position_embeddings=cfg["max_position"], type_vocab_size=cfg["type_vocab"],
                layer_norm_eps=cfg["ln_eps"], pad_token_id=0, hidden_act="gelu"))
            hf.load_state_dict(sd, strict=False)
            self.model = hf.eval()

    def describe(self) -> str:
        if self.kind == "reference":
            return ("baseline/_ref/MLM_PLL/main.py (unmodified) set_dataloader + run_one_epoch(train_mode=False, "
                    "do_scoring=True) on transformers.BertForMaskedLM, batch 32, num_worker 0, fp32")
        return "oracle port of MLM_PLL/main.py run_one_epoch (baseline/_ref absent), batch 32, fp32"

    def run(self, tok, off, n_hyps):
        """-> (hyps/s, seconds, masked copies, {hyp: PLL})."""
        import torch
        from oracle import pll_oracle
        hyps = {"u": {f"hyp_{i + 1}": [int(t) for t in tok[off[i]:off[i + 1]]] for i in range(n_hyps)}}
        copies = int(off[n_hyps] - off[0])
        t0 = time.perf_counter()
        if self.kind == "reference":
            rows, skel = [], {"u": {}}
            for h, toks in hyps["u"].items():
                skel["u"][h] = 0
                rows += pll_oracle.expand_rows(toks, "u", h)      # the a1 row schema (preprocess.py:9-30)
            loader = self.ref_main.set_dataloader(SimpleNamespace(batch_size=32, num_worker=0),
                                                  self.ref_main.MyDataset(rows), True)
            with torch.no_grad():
                out = self.ref_main.run_one_epoch(config=SimpleNamespace(device="cpu"), model=self.model,
                                                  dataloader=loader, output_score=skel, train_mode=False,
                                                  do_scoring=True)
        else:
            out = pll_oracle.score_hyps(self.sd, self.cfg, hyps, batch_size=32)   # score.yaml:16 batch_size
        dt = time.perf_counter() - t0
        return n_hyps / dt, dt, copies, out["u"]


def cpu_combiner(nb, lm, n_best):
    """The reference's find_best_weight (rescore.py:25-45) on the whole list -> (hyps/s, s, kind, weight, cer)."""
    ref_rescore = _load_reference_module("ref_rescore", "rescore.py", ".")
    am_l, lm_l = nb.am.tolist(), lm.tolist()
    cfg = SimpleNamespace(n_best=n_best)
    t0 = time.perf_counter()
    with np.errstate(all="ignore"):
        if ref_rescore is not None:
            bw, bc = ref_rescore.find_best_weight(am_l, lm_l, nb.hyps, nb.refs, cfg)
            kind = "reference"
        else:
            from oracle import rescore_oracle
            bw, bc = rescore_oracle.find_best_weight(am_l, lm_l, nb.hyps, nb.refs, cfg)
            kind = "port"
    dt = time.perf_counter() - t0
    return len(nb.hyps) * n_best / dt, dt, kind, float(bw), float(bc)


def auto_cpu_sample(args, wl) -> int:
    if args.cpu_sample_hyps:
        return args.cpu_sample_hyps
    per_step = 24 if wl["model"] == "bert-large-shaped" else 400
    if args.impl == "reference":                     # K timed steps must still end within a few minutes
        per_step = max(per_step // 8, min(per_step, per_step * 6 // max(args.steps, 1)))
    return per_step


def make_workload(args, wl, seed=0):
    from asr_rescoring_b200 import synth
    n_utts = args.utts or wl.get("sample_utts") or wl["n_utts"]
    return synth.make_nbest(n_utts, wl["n_best"], seed=seed, min_len=wl["min_len"], max_len=wl["max_len"]), n_utts


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on bounded samples."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from asr_rescoring_b200 import synth
    wl = WORKLOADS[args.workload]
    scaling = args.scaling or ("strong" if args.gpus > 1 else "weak")
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "data": "synthetic", "gpu_launches": 0}
    if wl["model"] is None:                              # c5: combiner only, whole list per step
        nb, n_utts = make_workload(args, wl)
        lm = synth.synthetic_lm_scores(nb, seed=1)
        times = []
        for i in range(min(args.warmup, 1) + args.steps):
            v, dt, kind, bw, bc = cpu_combiner(nb, lm, wl["n_best"])
            if i >= min(args.warmup, 1):
                times.append(dt)
        ms = 1e3 * float(np.mean(times))
        value = n_utts * wl["n_best"] / (ms / 1e3)
        sample = (f"the whole list ({n_utts} utterances x {wl['n_best']}-best x 101 weights) per step: "
                  f"rescore.find_best_weight from baseline/_ref under the jiwer stand-in (C Levenshtein)"
                  if kind == "reference" else "oracle port of rescore.find_best_weight (pure-Python Levenshtein)")
        _emit({**base, "value": value, "ms_per_step": ms, "dtype": "f64",
               "config": {"workload": wl["desc"], "n_best": wl["n_best"], "sample": sample},
               "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample},
               "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "best_weight": bw, "best_cer": bc})
        return
    cfg = model_cfg(wl["model"])
    n = auto_cpu_sample(args, wl)
    nb = synth.make_nbest(max(n // wl["n_best"] + 1, 4), wl["n_best"], seed=0, min_len=wl["min_len"], max_len=wl["max_len"])
    tok, off = nb.packed_tokens()
    sd = synth.random_init_state_dict(cfg, 10)
    n = min(n, len(off) - 1)
    arm = CpuPllArm(cfg, sd)
    for _ in range(min(args.warmup, 1)):
        arm.run(tok, off, min(n, 8))
    times, copies = [], 0
    for _ in range(args.steps):
        _, dt, copies, _ = arm.run(tok, off, n)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = n / (ms / 1e3)
    sample = f"first {n} hypotheses ({copies} masked copies) of workload {args.workload} per step; {arm.describe()}"
    _emit({**base, "value": value, "ms_per_step": ms, "dtype": "f32",
           "config": {"workload": wl["desc"], "n_best": wl["n_best"], "sample": sample},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.threads, "kind": arm.kind, "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


_JSON_FD = None


def _claim_stdout():
    """Keep fd 1 for the JSON line only: everything else that writes to stdout during the run
    (NCCL's version banner, library chatter) is sent to stderr."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def _emit(line: dict):
    sys.stdout.flush()
    sys.stderr.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir: str, arrays: dict, limit: int = DUMP_LIMIT_BYTES):
    """arrays: {name: float32 / float64 ndarray} -> out_dir/<name>.npy.  When they exceed `limit` bytes
    together, an array larger than its equal share keeps a fixed, seeded sample of its last axis, and the
    sampled positions are written to out_dir/<name>_index.npy (float64), so the files stay within `limit`."""
    os.makedirs(out_dir, exist_ok=True)
    share = limit // max(len(arrays), 1)
    over = sum(a.nbytes for a in arrays.values()) > limit
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if over and a.nbytes > share:
            per_position = a.nbytes // a.shape[-1] + 8            # the values at one position + its index
            idx = np.sort(np.random.default_rng(0).choice(a.shape[-1], size=share // per_position, replace=False))
            a = a[..., idx]
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------------------------ GPU arm
def main(argv=None):
    args = parse_args(argv)
    _claim_stdout()
    wl = WORKLOADS[args.workload]
    if args.operand_dtype is None:
        args.operand_dtype = wl["dtype"] if wl["model"] else None
    if wl.get("sample_utts") and not args.utts:
        print(f"bench: workload {args.workload} runs on the first {wl['sample_utts']} utterances unless --utts is given "
              f"(the full list is minutes per pass); operand dtype {args.operand_dtype}", file=sys.stderr)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from asr_rescoring_b200 import _lib, engine, shard, synth

    rank, world, local = shard.dist_env()
    if world > 1:
        shard.init_process_group("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load()
    _lib.require_device()
    scaling = (args.scaling or "strong") if world > 1 else "weak"
    strong = world > 1 and scaling == "strong"
    combiner_only = wl["model"] is None
    n_best = wl["n_best"]

    # ------------------------------------------------------------------ workload and its shard
    nb, n_utts = make_workload(args, wl, seed=0 if (strong or world == 1) else rank)
    lens_all = np.array([[len(h) for h in hs] for hs in nb.hyps], np.int64)
    if strong:
        if combiner_only:                           # stage 4 alone: contiguous utterance blocks (rescore.sweep)
            parts = [np.arange(*shard.block_range(n_utts, r, world)) for r in range(world)]
        else:                                       # BASELINE configs[2]: LPT on the expanded-token cost
            parts = shard.lpt_partition(shard.utterance_costs(lens_all), world)
        utt_sel = parts[rank]
        loads = [int((lens_all[p] * (lens_all[p] + 2)).sum()) for p in parts]
        counts_per_rank = [len(p) * n_best for p in parts]
    else:
        utt_sel = np.arange(n_utts)
        loads = [int((lens_all * (lens_all + 2)).sum())]
        counts_per_rank = [n_utts * n_best] * world
    n_total = n_utts * n_best if (strong or world == 1) else world * n_utts * n_best
    hyps = [nb.hyps[u] for u in utt_sel]
    refs = [nb.refs[u] for u in utt_sel]
    am = np.ascontiguousarray(nb.am[utt_sel])
    flat = [h for hs in hyps for h in hs]
    N, n_hyp = len(hyps), len(flat)
    # global (utterance-major) index of every local hypothesis: where its score lands after the gather
    global_idx = (shard.global_hyp_index(utt_sel, n_best) if (strong or world == 1)
                  else np.arange(n_hyp, dtype=np.int64) + rank * n_hyp)
    off = np.zeros(n_hyp + 1, np.int64)
    np.cumsum([len(h) for h in flat], out=off[1:])
    tok = np.fromiter((synth.synthetic_token_id(c) for h in flat for c in h), np.int32, int(off[-1]))
    lens = np.diff(off)
    hyp_len = lens.reshape(N, n_best).astype(np.int64)
    rc, ro = engine.pack_strings(refs)
    hc, ho = engine.pack_strings(flat)
    pair_ref = np.repeat(np.arange(N, dtype=np.int32), n_best)
    weights = np.arange(0.0, 1.01, 0.01)
    W = len(weights)
    ref_len_local = int(ro[-1])
    max_len = int(lens.max()) if n_hyp else 0

    scorer = cfg = sd = None
    if not combiner_only:
        cfg = model_cfg(wl["model"])
        sd = synth.random_init_state_dict(cfg, 10)
        scorer = engine.PllScorer(sd, cfg, device=local, max_chunk_tokens=args.chunk_tokens,
                                  operand_dtype=args.operand_dtype)
        lm_host = None
    else:
        lm_full = synth.synthetic_lm_scores(nb, seed=1)
        lm_host = np.ascontiguousarray(lm_full[utt_sel])

    # ------------------------------------------------------------------ device-resident inputs (`value`)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_tok, d_am, d_len = t(tok), t(am), t(hyp_len)
    d_rc, d_ro, d_hc, d_ho, d_pr, d_w = t(rc), t(ro), t(hc), t(ho), t(pair_ref), t(weights)
    n_max = max(counts_per_rank)
    d_pll_pad = torch.zeros(n_max, dtype=torch.float64, device=dev)         # local scores, padded for the gather
    d_pll = d_pll_pad[:n_hyp]
    if combiner_only:
        d_pll.copy_(t(lm_host.reshape(-1)))
    d_gather = torch.zeros(world * n_max, dtype=torch.float64, device=dev) if strong else None
    d_dist = torch.zeros(max(n_hyp, 1), dtype=torch.int32, device=dev)
    d_arg = torch.zeros(W * max(N, 1), dtype=torch.int32, device=dev)
    d_counts = torch.zeros(W + 1, dtype=torch.int64, device=dev)            # per-weight edit sums | reference length
    d_counts[W] = ref_len_local
    d_counts_all = torch.zeros_like(d_counts)
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)
    ev_lev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def stage4_device(time_lev=False):
        if time_lev:
            ev_lev[0].record(stream)
        _lib.check(lib.pllb_levenshtein(P(d_rc), P(d_ro), P(d_hc), P(d_ho), P(d_pr), n_hyp, max_len, P(d_dist), sp))
        if time_lev:
            ev_lev[1].record(stream)
        _lib.check(lib.pllb_rescore_sweep(P(d_am), P(d_pll), P(d_len), P(d_dist), N, n_best, P(d_w), W, 0,
                                          P(d_arg), P(d_counts), sp))
        if strong:                                   # reduce CER counts (rescore.py:40 is a corpus-level sum)
            d_counts_all.copy_(d_counts)
            dist.all_reduce(d_counts_all, op=dist.ReduceOp.SUM)

    def step_device(time_lev=False):
        if not combiner_only:
            scorer.score_device(d_tok, off, out=d_pll)
            if strong:                               # gather per-hypothesis scores (NCCL over NVLink)
                dist.all_gather_into_tensor(d_gather, d_pll_pad)
        stage4_device(time_lev)

    # ------------------------------------------------------------------ host buffers (`e2e`)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    h_tok, h_am, h_len = pin(tok), pin(am), pin(hyp_len)
    e2e_parts = {}

    def _acc(name, dt):
        e2e_parts[name] = e2e_parts.get(name, 0.0) + dt

    if combiner_only:
        from asr_rescoring_b200 import rescore as dropin
        am_l, lm_l = am.tolist(), lm_host.tolist()
        am_full_l, lm_full_l = nb.am.tolist(), lm_full.tolist()
        dcfg = SimpleNamespace(n_best=n_best)

        def step_host():
            t0 = time.perf_counter()
            if strong:      # the product's sharded sweep on this rank's block (block partition == utt_sel)
                _, cers, _ = dropin.sweep(am_full_l, lm_full_l, nb.hyps, nb.refs, dcfg)
                res = (float(weights[int(np.argmin(cers))]), float(cers.min()))
            else:
                res = dropin.find_best_weight(am_l, lm_l, hyps, refs, dcfg)
            _acc("rescore.find_best_weight", time.perf_counter() - t0)
            return None, res
    else:
        def step_host():
            t0 = time.perf_counter()
            pll = scorer.score_packed(h_tok, off)
            t1 = time.perf_counter()
            if strong:
                full = shard.gather_scores(pll, global_idx, n_total)
            else:
                full = pll
            t2 = time.perf_counter()
            dist_h = engine.levenshtein_packed(rc, ro, hc, ho, pair_ref).reshape(N, n_best)
            t3 = time.perf_counter()
            arg, es = engine.rescore_sweep(h_am, pll.reshape(N, n_best), h_len, dist_h, weights, "B")
            counts = np.concatenate([es, [ref_len_local]]).astype(np.int64)
            if strong:
                counts = shard.reduce_counts(counts)
            t4 = time.perf_counter()
            _acc("pllb_score_host", t1 - t0); _acc("gather_scores", t2 - t1)
            _acc("pllb_levenshtein_host", t3 - t2); _acc("pllb_rescore_sweep_host+reduce_counts", t4 - t3)
            return full, counts

    if combiner_only:
        h2d = rc.nbytes + ro.nbytes + hc.nbytes + ho.nbytes + pair_ref.nbytes + am.nbytes + n_hyp * 8 + hyp_len.nbytes + \
            n_hyp * 4 + weights.nbytes
        d2h = n_hyp * 4 + W * N * 4 + W * 8
    else:
        h2d = tok.nbytes + (rc.nbytes + ro.nbytes + hc.nbytes + ho.nbytes + pair_ref.nbytes) + \
            (am.nbytes + n_hyp * 8 + hyp_len.nbytes + n_hyp * 4 + weights.nbytes) + 3 * 4 * (n_hyp + 64)
        d2h = n_hyp * 8 + n_hyp * 4 + W * N * 4 + W * 8

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def in_global_order(gathered):
        """The device gather (rank-major, padded to n_max) laid out in global hypothesis order."""
        g = gathered.reshape(world, n_max)
        full = np.zeros(n_total, np.float64)
        for r in range(world):
            full[shard.global_hyp_index(parts[r], n_best)] = g[r, :counts_per_rank[r]]
        return full

    # ------------------------------------------------------------------ value (device resident)
    for _ in range(args.warmup):
        step_device()
    barrier()
    if scorer:
        scorer.reset_stats()
        scorer.set_timing(False)
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    ms_value = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop()
    last_step = None
    if args.dump_outputs and rank == 0:              # the last timed step's results, copied after the timed region
        last_step = {"distance": d_dist[:n_hyp].cpu().numpy().astype(np.float32),
                     "argmax": d_arg[:W * N].cpu().numpy().reshape(W, N).astype(np.float32),
                     "edit_sums": (d_counts_all if strong else d_counts)[:W].cpu().numpy().astype(np.float64)}
        if not combiner_only:
            last_step = {"pll": in_global_order(d_gather.cpu().numpy()) if strong else d_pll.cpu().numpy(), **last_step}
    launches = 2 * args.steps + (int(scorer.stats()["kernel_launches"]) if scorer else 0)

    # one extra, untimed-for-`value` step with per-launch CUDA events: the per-kind GEMM breakdown
    st = None
    if scorer:
        scorer.reset_stats()
        scorer.set_timing(True)
    step_device(time_lev=True)
    barrier()
    lev_ms = ev_lev[0].elapsed_time(ev_lev[1])
    if scorer:
        st = scorer.stats()
        scorer.set_timing(False)
    es_dev = (d_counts_all if strong else d_counts).cpu().numpy()

    # ------------------------------------------------------------------ e2e (host buffers)
    for _ in range(min(args.warmup, 1)):
        step_host()
    barrier()
    e2e_parts.clear()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        full_host, counts_host = step_host()
    barrier()
    ms_e2e = 1e3 * (time.perf_counter() - t0) / args.steps

    # ------------------------------------------------------------------ checks + max over ranks
    checks = {}
    if not combiner_only:
        if strong:
            full_dev = in_global_order(d_gather.cpu().numpy())
            checks["device_gather_equals_host_gather"] = bool(np.array_equal(full_dev, full_host))
        else:
            full_dev = d_pll.cpu().numpy()
            checks["device_scores_equal_host_scores"] = bool(np.array_equal(full_dev, full_host))
        checks["edit_sums_device_equal_host"] = bool(np.array_equal(es_dev, counts_host))
        pll_checksum = float(np.sum(full_dev)) if (strong or world == 1) else None
        best_weight = float(weights[int(np.argmin(es_dev[:W]))])
        best_cer = float(es_dev[:W].min()) / float(es_dev[W])
    else:
        pll_checksum = None
        best_weight = float(weights[int(np.argmin(es_dev[:W]))])
        best_cer = float(es_dev[:W].min()) / float(es_dev[W])
        checks["find_best_weight_equals_device_sweep"] = bool(counts_host[0] == best_weight and counts_host[1] == best_cer)

    stats = torch.tensor([ms_value, ms_e2e, float(n_hyp)], dtype=torch.float64, device=dev)
    if world > 1:
        mx, mn, sm = stats.clone(), stats.clone(), stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_value_min, ms_value, ms_e2e, total_hyps = float(mn[0]), float(mx[0]), float(mx[1]), float(sm[2])
        if st:                                       # per-rank device time of the scoring call alone (the last, timed step)
            tt = torch.tensor([st["last_total_ms"]], dtype=torch.float64, device=dev)
            tl = [torch.zeros_like(tt) for _ in range(world)]
            dist.all_gather(tl, tt)
            score_ms_by_rank = [float(x) for x in tl]
        else:
            score_ms_by_rank = None
    else:
        ms_value_min, total_hyps = ms_value, float(n_hyp)
        score_ms_by_rank = [st["last_total_ms"]] if st else None

    out = None
    if rank == 0:
        peak_tf, peak_hbm, peak_src = peaks()
        config = {"workload": wl["desc"], "utterances_total": n_utts if (strong or world == 1) else world * n_utts,
                  "utterances_per_gpu": N if not strong else [len(p) for p in parts], "n_best": n_best,
                  "hyps_rank0": n_hyp, "weights_grid": W, "parallelism": f"utterance-sharded x{world}",
                  "partition": ("LPT on sum L(L+2)" if not combiner_only else "contiguous utterance blocks") if strong else "replica per rank",
                  "lpt_load_imbalance": (max(loads) / (sum(loads) / len(loads)) - 1.0) if strong else 0.0,
                  "collectives_in_timed_region": (["all_gather(scores)", "all_reduce(edit sums + ref length)"]
                                                  if strong and not combiner_only else
                                                  ["all_reduce(edit sums + ref length)"] if strong else []),
                  "step_ms_min_over_ranks": ms_value_min, "step_ms_max_over_ranks": ms_value,
                  "score_call_ms_by_rank": score_ms_by_rank}
        out = {"metric": METRIC, "value": total_hyps / (ms_value / 1e3), "unit": UNIT, "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_value, "higher_is_better": True,
               "scaling": scaling, "vs_baseline": None, "dtype": args.operand_dtype or "f64", "data": "synthetic",
               "config": config,
               "e2e": {"value": total_hyps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                       "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e,
                       "ms_parts": {k: 1e3 * v / args.steps for k, v in e2e_parts.items()}},
               "gpu_launches": launches, "clocks": clocks, "checks": checks,
               "best_weight": best_weight, "best_cer": best_cer}
        if pll_checksum is not None:
            out["pll_checksum"] = pll_checksum
        if combiner_only:
            lev_bytes = rc.nbytes + ro.nbytes + hc.nbytes + ho.nbytes + pair_ref.nbytes + 4 * n_hyp
            ach = lev_bytes / (lev_ms / 1e3) / 1e9 if lev_ms > 0 else None
            config["l2"] = "inputs (a few MB) are L2-resident by design; the kernels are latency/compute-bound"
            out["roofline"] = {"bound": "hbm", "kernel": "levenshtein_kernel", "achieved": ach, "peak": peak_hbm,
                               "unit": "GB/s", "frac": (ach / peak_hbm) if ach else None, "traffic": None,
                               "peak_source": peak_src, "kernel_ms": lev_ms, "algorithmic_bytes_per_launch": lev_bytes,
                               "note": "integer DP over <= 64-character strings: bounded by dependent-issue latency, "
                                       "not by bytes; the fraction is reported, not claimed as a roofline"}
        else:
            config.update({"masked_copies_rank0": int(lens.sum()), "packed_tokens_rank0": int((lens * (lens + 2)).sum()),
                           "chunk_tokens": args.chunk_tokens,
                           "l2": "activations per chunk (>= 15 GB) exceed L2; no flush needed",
                           "algorithmic_tflop_per_step_rank0": total_flops(lens, cfg) / 1e12})
            ms_k, fl_k = st["gemm_ms_by_kind"], st["gemm_flops_by_kind"]
            H = cfg["hidden"]
            by_kind = {}
            for k in ms_k:
                if ms_k[k] <= 0:
                    continue
                tf = fl_k[k] / (ms_k[k] / 1e3) / 1e12
                by_kind[k] = {"kernel": KIND_KERNEL[k], "ms": ms_k[k], "tflop": fl_k[k] / 1e12, "tflops": tf,
                              "frac_tensor": tf / peak_tf}
            if "attn_out" in by_kind:
                # HBM-bound (AI 128 FLOP/B): per row fp32 residual in + out, 16-bit A in, 16-bit copy out = 12H bytes
                rows_ao = fl_k["attn_out"] / (2.0 * H * H)
                gbs = rows_ao * 12 * H / (ms_k["attn_out"] / 1e3) / 1e9
                by_kind["attn_out"].update({"bound": "hbm", "algorithmic_gb": rows_ao * 12 * H / 1e9, "gbs": gbs,
                                            "frac_hbm": gbs / peak_hbm})
            dom = max(by_kind, key=lambda k: by_kind[k]["ms"])
            gemm_ms = st["last_gemm_ms"]
            fam = st["gemm_flops"] / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
            traffic, tsrc = None, None
            tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
            if os.path.exists(tp):
                tj = json.load(open(tp))
                traffic = tj.get("by_kind_dram_bytes_per_launch", {}).get(dom, tj.get("gemm_dram_bytes_per_launch"))
                tsrc = ("profile constant: dram__bytes_read.sum + dram__bytes_write.sum per launch from one "
                        "`ncu --set full` capture (profiles/roofline_traffic.json), not measured by this run")
            out["roofline"] = {"bound": "tensor", "kernel": KIND_KERNEL[dom], "kind": dom,
                               "achieved": by_kind[dom]["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
                               "frac": by_kind[dom]["frac_tensor"], "traffic": traffic, "traffic_source": tsrc,
                               "peak_source": peak_src, "share_of_step": by_kind[dom]["ms"] / st["last_total_ms"],
                               "by_kind": by_kind,
                               "gemm_family": {"achieved": fam, "frac": fam / peak_tf if fam else None,
                                               "launches_per_step": int(st["last_gemm_launches"]), "ms_per_step": gemm_ms,
                                               "share_of_score_call": gemm_ms / st["last_total_ms"],
                                               "executed_gemm_tflop_per_step": st["gemm_flops"] / 1e12,
                                               "survey_formula_gemm_tflop_per_step": gemm_flops(lens, cfg) / 1e12}}
            out["whole_step_tflops"] = (total_flops(lens_all if strong else lens, cfg) * (1 if strong or world == 1 else world)
                                        / (ms_value / 1e3) / 1e12)
        if world == 1 and not args.no_cpu_baseline:
            if combiner_only:
                v, dt, kind, bw, bc = cpu_combiner(nb, lm_full, n_best)
                out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
                                       "sample": f"the whole list, rescore.find_best_weight from baseline/_ref under the jiwer "
                                                 f"stand-in (C Levenshtein), {dt:.1f} s; best_weight {bw}, cer {bc}"}
                checks["cpu_reference_best_weight_and_cer_equal"] = bool(bw == best_weight and bc == best_cer)
            else:
                arm = CpuPllArm(cfg, sd)
                n_cpu = min(auto_cpu_sample(args, wl), n_hyp)
                v, dt, copies, ref_pll = arm.run(tok, off, n_cpu)
                got = full_dev[global_idx[:n_cpu]] if (strong or world == 1) else full_dev[:n_cpu]
                err = np.abs(np.array([ref_pll[f"hyp_{i + 1}"] for i in range(n_cpu)]) - got)
                out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": arm.threads, "kind": arm.kind,
                                       "sample": f"first {n_cpu} hypotheses ({copies} masked copies) of the same workload; "
                                                 f"{arm.describe()}; {dt:.1f} s",
                                       "max_abs_dpll_vs_gpu": float(err.max()), "mean_abs_dpll_vs_gpu": float(err.mean())}
        if last_step is not None:
            write_outputs(args.dump_outputs, last_step)
    if scorer:
        scorer.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        _emit(out)                             # the JSON line is the only thing on stdout


if __name__ == "__main__":
    main()
