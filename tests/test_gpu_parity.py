"""Parity of the CUDA path (through the C ABI of libpllb200.so) against the oracle and the
committed golden fixtures.  Integer / byte / fp64 work: bit-exact.  PLL: within 0.05 nats
absolute per hypothesis (north_star: bf16 operands, fp32 accumulate)."""
import json
import os

import numpy as np
import pytest

import oracle
from oracle import pll_oracle, rescore_oracle
from asr_rescoring_b200 import engine, synth

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("require_gpu")]

PLL_TOL = 0.05   # nats, absolute, per hypothesis (BASELINE.json north_star)


# ----------------------------------------------------------------------------- stage 4
def test_levenshtein_reference_kats_bit_exact(gold_dir):
    z = np.load(os.path.join(gold_dir, "levenshtein_kat.npz"))
    got = engine.levenshtein_packed(z["ref_cp"], z["ref_off"], z["hyp_cp"], z["hyp_off"],
                                    np.arange(len(z["dist"]), dtype=np.int32))
    assert np.array_equal(got, z["dist"])           # Nbest_Align/cer.json, 7 176 pairs
    assert int(got.sum()) == 3230


@pytest.mark.parametrize("n", [0, 1, 2, 31, 32, 33, 63, 64, 65, 128, 129, 300, 513, 1024])
def test_levenshtein_lengths_and_edge_cases(n):
    rng = np.random.default_rng(n)
    mk = lambda k: "".join(chr(0x4E00 + int(c)) for c in rng.integers(0, 12, size=k))
    refs = [mk(max(n + int(rng.integers(-5, 6)), 0)) for _ in range(40)] + ["", mk(n), mk(3)]
    hyps = [mk(n) for _ in range(40)] + [mk(n), "", ""]
    hyps[0] = refs[0][:1024]
    assert np.array_equal(engine.levenshtein(refs, hyps), oracle.levenshtein_strings(refs, hyps))


def test_levenshtein_rejects_too_long():
    from asr_rescoring_b200._lib import PllbError
    with pytest.raises(PllbError):
        engine.levenshtein(["a"], ["b" * 1025])


def test_levenshtein_pair_ref_and_strip():
    refs = ["你好嗎", "how are you"]
    hyps = ["你好不好", " 你好嗎 ", "how are you doing", "haw are you"]
    got = engine.levenshtein(refs, hyps, pair_ref=[0, 0, 1, 1])
    assert got.tolist() == [2, 0, 6, 1]             # align.py:13-18 example 2 has distance 2


def _bits_equal(a, b):
    return bool(((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))).all())


def test_combiner_bit_exact_vs_reference_golden(gold_dir):
    z = np.load(os.path.join(gold_dir, "combiner_golden.npz"))
    N, nb = z["am"].shape
    pair_ref = np.repeat(np.arange(N, dtype=np.int32), nb)
    dist = engine.levenshtein_packed(z["ref_cp"], z["ref_off"], z["hyp_cp"], z["hyp_off"], pair_ref).reshape(N, nb)
    assert np.array_equal(dist, oracle.levenshtein_batch(z["ref_cp"], z["ref_off"], z["hyp_cp"], z["hyp_off"], pair_ref).reshape(N, nb))
    arg, es = engine.rescore_sweep(z["am"], z["lm"], z["lens"], dist, z["weights"], "B")
    assert np.array_equal(arg, z["argmax"])         # rescore.py outputs, incl. tie and NaN rows
    for i, wi in enumerate(z["score_idx"]):
        s = engine.rescore_scores(z["am"], z["lm"], z["lens"], z["weights"][wi], "B")
        assert _bits_equal(s, z["scores"][i])
    cers = es / float(z["ref_off"][-1])
    assert z["weights"][int(np.argmin(cers))] == float(z["best_weight"]) and cers.min() == float(z["best_cer"])


@pytest.mark.parametrize("variant,code", [("B", 0), ("A", 1), ("C", 2)])
def test_combiner_variants_vs_oracle(variant, code):
    nb = synth.make_nbest(400, 7, seed=21)
    lm = synth.synthetic_lm_scores(nb, seed=5)
    lens = np.array([[len(h) for h in hs] for hs in nb.hyps], np.int64)
    lens[3, 2] = 0                                   # len == 0 -> inf / nan semantics (rescore.py:51)
    rng = np.random.default_rng(0)
    dist = rng.integers(0, 9, size=lens.shape).astype(np.int32)
    w = np.arange(0.0, 1.01, 0.01)
    arg, es = engine.rescore_sweep(nb.am, lm, lens, dist, w, variant)
    arg_o, es_o = oracle.rescore_sweep(nb.am, lm, lens, dist, w, code)
    assert np.array_equal(arg, arg_o) and np.array_equal(es, es_o)
    with np.errstate(all="ignore"):
        s_np = rescore_oracle.rescore(w[29], lens, nb.am, lm, rescore_oracle.config(7), variant)
    assert _bits_equal(engine.rescore_scores(nb.am, lm, lens, w[29], variant), s_np)


def test_drop_in_rescore_functions_match_oracle():
    from asr_rescoring_b200 import rescore as dropin
    nb = synth.make_nbest(200, 10, seed=33)
    lm = synth.synthetic_lm_scores(nb, seed=6)
    cfg = rescore_oracle.config(6)                   # n_best < available: am is sliced, lm pre-sliced (rescore.py:48-49)
    lm6 = [r[:6] for r in lm.tolist()]
    bw, bc = dropin.find_best_weight(nb.am.tolist(), lm6, nb.hyps, nb.refs, cfg)
    bw_o, bc_o = rescore_oracle.find_best_weight(nb.am.tolist(), lm6, nb.hyps, nb.refs, cfg)
    assert bw == bw_o and bc == bc_o
    lens = dropin._hyps_len(nb.hyps, 6)
    s = dropin.rescore(bw, lens, nb.am.tolist(), lm6, cfg)
    assert _bits_equal(s, rescore_oracle.rescore(bw_o, lens, nb.am.tolist(), lm6, cfg))
    assert dropin.get_highest_score_hyp(s, nb.hyps) == rescore_oracle.get_highest_score_hyp(s, nb.hyps)
    assert dropin.cer(nb.refs, [h[0] for h in nb.hyps]) == rescore_oracle.cer(nb.refs, [h[0] for h in nb.hyps])
    with pytest.raises(ValueError):
        dropin.cer([""], ["a"])


def test_other_cer_call_sites_match_oracle():
    """espnet_data/preprocess/main.py:59-60 (hyps_cer.json) and RMBR's CER utility / mbr_decode."""
    import torch
    from asr_rescoring_b200 import cer_clients
    nb = synth.make_nbest(40, 6, seed=44)
    got = cer_clients.hyps_cer(nb.hyps_text(), nb.ref_text())
    for u, r, hs in zip(nb.utt_ids, nb.refs, nb.hyps):
        for k, h in enumerate(hs):
            assert got[u][f"hyp_{k + 1}"] == rescore_oracle.cer(r, h)
    with pytest.raises(ValueError):
        cer_clients.pair_cer([" "], ["a"])

    class OracleCer(cer_clients.BaseFunction):           # RMBR/utility_functions.py:24-33 on the oracle
        def score(self, cands, refs):
            return [1 - rescore_oracle.cer(r, c) for c, r in zip(cands, refs)]

    pred, sc = cer_clients.mbr_decode(5, nb.hyps, cer_clients.CerScoreFunction(None))
    pred_o, sc_o = cer_clients.mbr_decode(5, nb.hyps, OracleCer(None))
    assert pred == pred_o and torch.equal(sc, sc_o)


def test_combiner_full_size_properties():
    """Config 5 size (7 176 x 50-best, 101 weights): size-independent properties."""
    nb = synth.make_nbest(7176, 50, seed=9)
    lm = synth.synthetic_lm_scores(nb, seed=3)
    lens = np.array([[len(h) for h in hs] for hs in nb.hyps], np.int64)
    from asr_rescoring_b200 import rescore as dropin
    dist = dropin.pair_distances(nb.hyps, nb.refs, 50)
    assert dist.shape == (7176, 50)
    # bounded by the number of random edits applied; 0 iff strings equal
    assert (dist <= nb.edits).all()
    same = np.array([[h == r for h in hs] for hs, r in zip(nb.hyps, nb.refs)])
    assert ((dist == 0) == same).all()
    w = np.arange(0.0, 1.01, 0.01)
    arg, es = engine.rescore_sweep(nb.am, lm, lens, dist, w, "B")
    # weight 0 -> argmax of am/len; weight 1 (last grid point is 1.0) -> argmax of lm/len
    assert np.array_equal(arg[0], np.argmax(nb.am / lens, axis=1))
    assert w[-1] == 1.0 and np.array_equal(arg[-1], np.argmax((1 - w[-1]) * nb.am / lens + w[-1] * lm / lens, axis=1))
    # checksum of checksums: edit sums equal the gathered distances, any order
    assert np.array_equal(es, np.take_along_axis(dist, arg.T.astype(np.int64), axis=1).sum(0))
    # sample of rows against the C oracle
    rows = np.arange(0, 7176, 97)
    arg_o, _ = oracle.rescore_sweep(nb.am[rows], lm[rows], lens[rows], dist[rows], w, 0)
    assert np.array_equal(arg[:, rows], arg_o)


# ----------------------------------------------------------------------------- stage 1
def test_expansion_matches_reference_rows():
    sd = synth.random_init_state_dict(synth.BERT_TINY, 1)
    with engine.PllScorer(sd, synth.BERT_TINY) as sc:
        nb = synth.make_nbest(30, 6, seed=1)
        nb.hyps[0][0] = ""                           # empty hypothesis -> no rows
        nb.hyps[2][3] = nb.hyps[2][3][:1]            # single token
        tok, off = nb.packed_tokens(synth.BERT_TINY["vocab"])
        ids, mp, lab = sc.expand(tok, off)
        ids_o, mp_o, lab_o = oracle.expand(tok, off)
        assert np.array_equal(ids, ids_o) and np.array_equal(mp, mp_o) and np.array_equal(lab, lab_o)


# ----------------------------------------------------------------------------- GEMM
@pytest.mark.parametrize("M,N,K", [(1, 256, 64), (127, 256, 64), (128, 512, 128), (300, 768, 768), (1000, 2304, 768),
                                   (2049, 3072, 768), (513, 768, 3072), (700, 1024, 1024)])
def test_tcgen05_gemm_vs_fp32_torch(M, N, K):
    import torch
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda").bfloat16()
    W = (torch.randn(N, K, device="cuda") * 0.05).bfloat16()
    b = torch.randn(N, device="cuda")
    ref = A.float() @ W.float().T + b              # plain PyTorch fp32 reference of the same op
    for epi in (2, 3, 0, 1):
        out = engine.debug_gemm(A, W, b, epi).float()
        r = torch.nn.functional.gelu(ref) if epi in (1, 3) else ref
        if epi >= 2:
            assert (out - r).abs().max().item() < 1e-3
        else:                                        # bf16 output: half an ulp of the value
            assert ((out - r).abs() <= r.abs() * 2 ** -8 + 1e-3).all()
        simt = engine.debug_gemm(A, W, b, epi, simt=True).float()
        assert (out - simt).abs().max().item() < (1e-3 if epi >= 2 else 0.07)


# ----------------------------------------------------------------------------- encoder / PLL
def _oracle_hidden(sd, cfg, tok, off, upto):
    import torch
    out = []
    for h in range(len(off) - 1):
        toks = [int(t) for t in tok[off[h]:off[h + 1]]]
        for r in pll_oracle.expand_rows(toks, "u", "h"):
            ids = torch.tensor([r["input_ids"]])
            out.append(pll_oracle.bert_mlm_logits(sd, cfg, ids, torch.ones_like(ids), upto_layer=upto, return_hidden=True)[0])
    return torch.cat(out)


def test_embeddings_and_layers_vs_oracle():
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 10, perturb=True)
    nb = synth.make_nbest(4, 3, seed=2)
    tok, off = nb.packed_tokens(cfg["vocab"])
    with engine.PllScorer(sd, cfg) as sc:
        e0 = (sc.hidden(tok, off, 0) - _oracle_hidden(sd, cfg, tok, off, 0)).abs().max().item()
        assert e0 < 5e-6                              # fp32 embedding + LayerNorm
        for upto in (1, 2):
            err = (sc.hidden(tok, off, upto) - _oracle_hidden(sd, cfg, tok, off, upto)).abs()
            assert err.max().item() < 0.03 and err.mean().item() < 3e-3   # bf16 GEMM operands


@pytest.mark.parametrize("hidden", [256, 512, 768, 1024])
def test_fused_gemm_layernorm_cluster_sizes(hidden):
    """The residual+LayerNorm epilogue runs on a cluster of hidden/256 CTAs that exchange row
    statistics through distributed shared memory: every cluster size against the fp32 oracle,
    with a row count that is not a multiple of the 128-row tile and several tiles per cluster."""
    cfg = dict(num_layers=2, hidden=hidden, num_heads=hidden // 64, intermediate=2 * hidden, vocab=1200,
               max_position=64, type_vocab=2, ln_eps=1e-12)
    sd = synth.random_init_state_dict(cfg, 21, perturb=True)
    rng = np.random.default_rng(hidden)
    lens = [int(x) for x in rng.integers(1, 40, size=60)]
    off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rng.integers(104, cfg["vocab"], size=int(off[-1])).astype(np.int32)
    with engine.PllScorer(sd, cfg) as sc:
        got = sc.hidden(tok[:off[8]], off[:9], 2)
        pll = sc.score_packed(tok, off)
    exp = _oracle_hidden(sd, cfg, tok[:off[8]], off[:9], 2)
    err = (got - exp).abs()
    assert err.max().item() < 0.04 and err.mean().item() < 4e-3, (err.max().item(), err.mean().item())
    hyps = {"u": {f"hyp_{i + 1}": [int(t) for t in tok[off[i]:off[i + 1]]] for i in range(12)}}
    ref = pll_oracle.score_hyps(sd, cfg, hyps)
    for i in range(12):
        assert abs(pll[i] - ref["u"][f"hyp_{i + 1}"]) <= PLL_TOL


def test_attention_paths_short_and_long_sequences():
    """T <= 32 takes the cp.async-staged attention path, longer sequences the streaming one;
    both against the fp32 oracle after one full layer, incl. T = 3 and T = max_position."""
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 12, perturb=True)
    rng = np.random.default_rng(3)
    lens = [1, 2, 14, 15, 16, 29, 30, 31, 32, 47, 64, 100, cfg["max_position"] - 2]
    off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    tok = rng.integers(104, cfg["vocab"], size=int(off[-1])).astype(np.int32)
    with engine.PllScorer(sd, cfg) as sc:
        got = sc.hidden(tok, off, 1)
    exp = _oracle_hidden(sd, cfg, tok, off, 1)
    err = (got - exp).abs()
    assert err.max().item() < 0.03 and err.mean().item() < 3e-3, (err.max().item(), err.mean().item())


def test_pll_vs_reference_golden(gold_dir):
    gold = json.load(open(os.path.join(gold_dir, "pll_golden.json")))
    for case in gold["cases"]:
        sd = synth.random_init_state_dict(case["cfg"], case["seed"], case["perturb"])
        with engine.PllScorer(sd, case["cfg"]) as sc:
            got = sc.score_hyps(case["hyps"])
        for u, hs in case["pll"].items():
            for h, v in hs.items():
                assert abs(got[u][h] - v) <= PLL_TOL, (case["name"], u, h, got[u][h], v)
                if len(case["hyps"][u][h]) == 0:
                    assert got[u][h] == 0 and isinstance(got[u][h], int)


def test_pll_fp16_operand_mode_vs_reference_golden(gold_dir):
    """operand_dtype="fp16": same kernels with IEEE-half operands; the error against the
    reference drops ~6x (10 mantissa bits instead of 7)."""
    gold = json.load(open(os.path.join(gold_dir, "pll_golden.json")))
    for case in gold["cases"]:
        sd = synth.random_init_state_dict(case["cfg"], case["seed"], case["perturb"])
        with engine.PllScorer(sd, case["cfg"], operand_dtype="fp16") as sc:
            got = sc.score_hyps(case["hyps"])
        worst = max(abs(got[u][h] - v) for u, hs in case["pll"].items() for h, v in hs.items())
        assert worst <= 0.012, (case["name"], worst)


def test_pll_vs_live_oracle_and_rescored_one_best():
    cfg = synth.BERT_BASE_CHINESE
    sd = synth.random_init_state_dict(cfg, 10)
    nb = synth.make_nbest(12, 5, seed=77)
    tok, off = nb.packed_tokens()
    hyps, i = {}, 0
    for u, hs in zip(nb.utt_ids, nb.hyps):
        hyps[u] = {}
        for k in range(len(hs)):
            hyps[u][f"hyp_{k + 1}"] = [int(t) for t in tok[off[i]:off[i + 1]]]
            i += 1
    exp = pll_oracle.score_hyps(sd, cfg, hyps)
    with engine.PllScorer(sd, cfg) as sc:
        got = sc.score_hyps(hyps)
        pll, tl = sc.score_packed(tok, off, return_token_logp=True)
    d = np.array([got[u][h] - exp[u][h] for u in hyps for h in hyps[u]])
    assert np.abs(d).max() <= PLL_TOL, np.abs(d).max()
    # sum of the per-token terms (fp32) in order, in double, is the PLL (MLM_PLL/main.py:105-107)
    for j in range(len(off) - 1):
        assert pll[j] == float(np.sum(tl[off[j]:off[j + 1]].astype(np.float64)))
    # rescored 1-best at the weight the oracle picks
    lm_g = np.array([[got[u][h] for h in hyps[u]] for u in hyps])
    lm_o = np.array([[exp[u][h] for h in hyps[u]] for u in hyps])
    c = rescore_oracle.config(5)
    bw, _ = rescore_oracle.find_best_weight(nb.am.tolist(), lm_o.tolist(), nb.hyps, nb.refs, c)
    lens = rescore_oracle.hyps_len_of(nb.hyps, 5)
    a_o = np.argmax(rescore_oracle.rescore(bw, lens, nb.am, lm_o, c), -1)
    a_g = np.argmax(rescore_oracle.rescore(bw, lens, nb.am, lm_g, c), -1)
    assert (a_o == a_g).mean() >= 0.9


def test_config1_100x10_best_against_oracle_acceptance():
    """BASELINE.json configs[0] (100 utterances x 10-best, random-init bert-base-chinese) run in
    full through the oracle port of the reference's CPU path and through the GPU path:
    north_star acceptance — |dPLL| <= 0.05 nats per hypothesis, identical rescored 1-best,
    identical CER counts at the weight the reference picks."""
    cfg = synth.BERT_BASE_CHINESE
    sd = synth.random_init_state_dict(cfg, 10)
    nb = synth.make_nbest(100, 10, seed=0)
    tok, off = nb.packed_tokens()
    n = len(off) - 1
    hyps = {"u": {f"hyp_{i + 1}": [int(t) for t in tok[off[i]:off[i + 1]]] for i in range(n)}}
    exp = pll_oracle.score_hyps(sd, cfg, hyps)
    ref = np.array([exp["u"][f"hyp_{i + 1}"] for i in range(n)])
    with engine.PllScorer(sd, cfg) as sc:
        got = sc.score_packed(tok, off)
    err = np.abs(got - ref)
    assert err.max() <= PLL_TOL, (err.max(), int((err > PLL_TOL).sum()))
    assert err.mean() < 0.02
    from asr_rescoring_b200 import rescore as dropin
    c = rescore_oracle.config(10)
    lm_o, lm_g = ref.reshape(100, 10).tolist(), got.reshape(100, 10).tolist()
    bw_o, cer_o = rescore_oracle.find_best_weight(nb.am.tolist(), lm_o, nb.hyps, nb.refs, c)
    bw_g, cer_g = dropin.find_best_weight(nb.am.tolist(), lm_g, nb.hyps, nb.refs, c)
    lens = rescore_oracle.hyps_len_of(nb.hyps, 10)
    a_o = np.argmax(rescore_oracle.rescore(bw_o, lens, nb.am, np.array(lm_o), c), -1)
    a_g = np.argmax(rescore_oracle.rescore(bw_o, lens, nb.am, np.array(lm_g), c), -1)
    assert (a_o == a_g).mean() >= 0.99, (a_o != a_g).sum()     # rescored 1-best at the reference's weight
    # CER counts with the oracle's PLLs through the GPU combiner are bit-exact
    bw_x, cer_x = dropin.find_best_weight(nb.am.tolist(), lm_o, nb.hyps, nb.refs, c)
    assert bw_x == bw_o and cer_x == cer_o
    assert abs(cer_g - cer_o) <= 2.0 / sum(len(r) for r in nb.refs)


def test_rescorebert_scoring_vs_reference_golden(gold_dir):
    """Sequence-level scoring ([CLS] -> Linear(H,1)) against the reference's RescoreBert.forward
    (tests/golden/rescorebert_golden.json) and the live oracle, incl. an empty hypothesis and
    multi-chunk packing."""
    import torch
    from asr_rescoring_b200.RescoreBert.model import RescoreBert
    gold = json.load(open(os.path.join(gold_dir, "rescorebert_golden.json")))
    for case in gold["cases"]:
        sd = synth.random_init_state_dict(case["cfg"], case["seed"], case["perturb"])
        sd = {k: v for k, v in sd.items() if k.startswith("bert.")}
        sd["linear.weight"] = torch.tensor(case["linear_w"]).reshape(1, -1)
        sd["linear.bias"] = torch.tensor([case["linear_b"]])
        lists = case["tokens"]
        off = np.zeros(len(lists) + 1, np.int64)
        np.cumsum([len(t) for t in lists], out=off[1:])
        tok = np.array([t for l in lists for t in l], np.int32)
        with RescoreBert(sd, case["cfg"], max_chunk_tokens=1024) as m:
            got = m.score_packed(tok, off)
            assert not m.encoder.has_mlm_head
            from asr_rescoring_b200._lib import PllbError
            with pytest.raises(PllbError):
                m.encoder.score_packed(tok, off)          # no MLM head in this checkpoint
        ref = np.array(case["scores"])
        # bf16 GEMM operands: the [CLS] state carries ~1e-2 absolute error, the head is a 768-term dot
        assert np.abs(got - ref).max() < 0.05, np.abs(got - ref).max()
        full = synth.random_init_state_dict(case["cfg"], case["seed"], case["perturb"])
        exp = pll_oracle.rescore_bert_scores(full, case["cfg"], lists, case["linear_w"], case["linear_b"])
        assert np.abs(got - np.array(exp)).max() < 0.05


def test_scoring_is_deterministic_and_chunking_invariant():
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 4, perturb=True)
    nb = synth.make_nbest(60, 5, seed=8)
    nb.hyps[5][1] = ""
    tok, off = nb.packed_tokens(cfg["vocab"])
    with engine.PllScorer(sd, cfg) as big, engine.PllScorer(sd, cfg, max_chunk_tokens=2048) as small:
        a, ta = big.score_packed(tok, off, return_token_logp=True)
        b = big.score_packed(tok, off)
        c, tc = small.score_packed(tok, off, return_token_logp=True)
        assert small.stats()["chunks"] > 5 and big.stats()["chunks"] == 2
    assert np.array_equal(a, b)                       # run twice: bitwise identical
    assert np.array_equal(a, c) and np.array_equal(ta, tc)   # any chunking: bitwise identical
    empty = np.diff(off) == 0
    assert (a[empty] == 0.0).all() and np.isfinite(a).all()


def test_duplicate_hypotheses_score_identically_at_scale():
    """Size-independent property at a multi-chunk size: a hypothesis' PLL does not depend on
    its neighbours or its position in the packed batch."""
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 5)
    nb = synth.make_nbest(400, 10, seed=12)
    tok, off = nb.packed_tokens(cfg["vocab"])
    L = np.diff(off)
    perm = np.random.default_rng(0).permutation(len(L))
    tok_p = np.concatenate([tok[off[i]:off[i + 1]] for i in perm])
    off_p = np.zeros(len(L) + 1, np.int64)
    np.cumsum(L[perm], out=off_p[1:])
    with engine.PllScorer(sd, cfg, max_chunk_tokens=1 << 16) as sc:
        a = sc.score_packed(tok, off)
        b = sc.score_packed(tok_p, off_p)
    assert np.array_equal(a[perm], b)


def test_too_long_hypothesis_is_rejected():
    from asr_rescoring_b200._lib import PllbError
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 5)
    with engine.PllScorer(sd, cfg) as sc:
        n = cfg["max_position"] - 1                  # needs n + 2 positions
        with pytest.raises(PllbError):
            sc.score_packed(np.full(n, 700, np.int32), np.array([0, n], np.int64))


def test_out_of_vocabulary_token_is_rejected():
    from asr_rescoring_b200._lib import PllbError
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 5)
    with engine.PllScorer(sd, cfg) as sc:
        for bad in (cfg["vocab"], -1):
            with pytest.raises(PllbError):
                sc.score_packed(np.array([700, bad, 701], np.int32), np.array([0, 3], np.int64))
        ok = sc.score_packed(np.array([700, cfg["vocab"] - 1, 701], np.int32), np.array([0, 3], np.int64))
        assert np.isfinite(ok).all()


def test_drop_in_run_one_epoch_matches_oracle_rows():
    from asr_rescoring_b200.MLM_PLL import main as dropin
    from types import SimpleNamespace
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 10, perturb=True)
    nb = synth.make_nbest(5, 3, seed=14)
    tok, off = nb.packed_tokens(cfg["vocab"])
    rows, i = [], 0
    for u, hs in zip(nb.utt_ids, nb.hyps):
        for k in range(len(hs)):
            rows += pll_oracle.expand_rows([int(t) for t in tok[off[i]:off[i + 1]]], u, f"hyp_{k + 1}")
            i += 1
    rows = rows[:len(rows) - 3]                      # num_of_data cuts the last hypothesis short
    skel = dropin.skeleton_from_rows(rows)
    exp = pll_oracle.score_rows(sd, cfg, rows, {u: dict(v) for u, v in skel.items()})
    with engine.PllScorer(sd, cfg) as sc:
        loader = dropin.set_dataloader(SimpleNamespace(batch_size=32, num_worker=5), dropin.MyDataset(rows), True)
        got = dropin.run_one_epoch(config=SimpleNamespace(device="cuda:0"), model=sc, dataloader=loader,
                                   output_score=skel, train_mode=False, do_scoring=True)
    for u in exp:
        for h in exp[u]:
            assert abs(got[u][h] - exp[u][h]) <= PLL_TOL


def test_drop_in_cli_end_to_end():
    """MLM_PLL/main.py --config score.yaml and rescore.py --config rescore.yaml as processes, on
    synthetic hyps_text / hyps_score / ref_text files, checked against the oracle."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "e2e_dropin.py")], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    assert "rescore.log matches the oracle" in out.stdout


def test_bench_dump_outputs_are_the_timed_results_and_repeat_across_runs(tmp_path):
    """bench.py --dump-outputs: what the last timed step computed, identical for 1 and 2 timed steps
    (seeded inputs), consistent with the JSON line, and the same scores as a direct scoring call."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lines = {}
    for steps in (1, 2):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "c1", "--steps", str(steps),
                              "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(steps))],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        lines[steps] = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
        assert lines[steps]["steps"] == steps
    names = ["argmax.npy", "distance.npy", "edit_sums.npy", "pll.npy"]
    assert sorted(os.listdir(tmp_path / "1")) == names == sorted(os.listdir(tmp_path / "2"))
    d = {n[:-4]: np.load(tmp_path / "2" / n) for n in names}
    for n in names:
        assert np.array_equal(np.load(tmp_path / "1" / n), d[n[:-4]]), n
    assert d["pll"].dtype == np.float64 and d["pll"].shape == (1000,) and d["argmax"].shape == (101, 100)
    assert d["distance"].dtype == np.float32 and d["edit_sums"].dtype == np.float64
    assert float(np.sum(d["pll"])) == lines[2]["pll_checksum"]
    assert float(np.arange(0.0, 1.01, 0.01)[int(np.argmin(d["edit_sums"]))]) == lines[2]["best_weight"]
    nb = synth.make_nbest(100, 10, seed=0)
    dist = oracle.levenshtein_strings([r for r in nb.refs for _ in range(10)], [h for hs in nb.hyps for h in hs])
    assert np.array_equal(d["distance"], dist.astype(np.float32))
    chosen = np.take_along_axis(dist.reshape(100, 10), d["argmax"].T.astype(np.int64), axis=1)
    assert np.array_equal(d["edit_sums"], chosen.sum(0).astype(np.float64))
    tok, off = nb.packed_tokens()
    with engine.PllScorer(synth.random_init_state_dict(synth.BERT_BASE_CHINESE, 10), synth.BERT_BASE_CHINESE,
                          operand_dtype=lines[2]["dtype"]) as sc:
        assert np.array_equal(sc.score_packed(tok, off), d["pll"])


def test_text_front_end_matches_the_host_tokenizer(tmp_path):
    """pllb_tokenize_host (+ host path for flagged hypotheses) == BertTokenizer-style encode, per string."""
    from asr_rescoring_b200.tokenizer import BertCharTokenizer, SyntheticCharTokenizer, encode_batch
    nb = synth.make_nbest(300, 10, seed=21)
    chars = sorted({c for r in nb.refs for c in r})
    vocab = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", "a", "ab", "##c", "##d", "hello", "1", "##2", ",", "。", "，", "?"] + chars[::2]
    vp = tmp_path / "vocab.txt"
    vp.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    strings = [h for hs in nb.hyps for h in hs]
    rng = np.random.default_rng(3)
    extra = ["", " ", "你好abc", "hello，世界", "abcd 12", "\x00" + strings[0] + "\ufffd", strings[1] + "\u3000" + strings[2],
             chr(0xF900) + strings[3], "。，?" + strings[4], chr(0x20000) + chr(0x2A700), "a\u0301" + strings[5], "あいう"]
    for i in rng.integers(0, len(strings), 40):                       # sprinkle whitespace / punctuation / Latin
        sidx = int(i)
        strings[sidx] = strings[sidx][:2] + str(rng.choice([" ", "，", "a", "\t", "12", "?"])) + strings[sidx][2:]
    strings += extra
    for tk in (BertCharTokenizer(str(vp)), SyntheticCharTokenizer()):
        ids, off = encode_batch(tk, strings)
        assert off[0] == 0 and len(off) == len(strings) + 1 and off[-1] == len(ids)
        for i, s_ in enumerate(strings):
            assert ids[off[i]:off[i + 1]].tolist() == tk.encode(s_), (type(tk).__name__, repr(s_))
    try:
        from transformers import BertTokenizer
        hf = BertTokenizer(str(vp))
    except Exception:
        hf = None
    if hf is not None:
        ids, off = encode_batch(BertCharTokenizer(str(vp)), strings)
        for i, s_ in enumerate(strings):
            assert ids[off[i]:off[i + 1]].tolist() == hf.convert_tokens_to_ids(hf.tokenize(s_)), repr(s_)
    # empty batch and all-flagged batch
    ids, off = encode_batch(SyntheticCharTokenizer(), [])
    assert len(ids) == 0 and off.tolist() == [0]
    ids, off = encode_batch(BertCharTokenizer(str(vp)), ["abc", "hello 12"])
    assert ids.tolist() == BertCharTokenizer(str(vp)).encode("abc") + BertCharTokenizer(str(vp)).encode("hello 12")


def test_back_to_back_async_calls_keep_their_own_metadata():
    """pllb_score is asynchronous on the caller's stream; three calls with different hypothesis
    sets issued without any synchronisation must each score their own input (the host-side
    metadata staging buffer is reused across calls)."""
    import torch
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 4)
    nbs = [synth.make_nbest(400, 10, seed=31), synth.make_nbest(30, 10, seed=32), synth.make_nbest(30, 10, seed=33)]
    packed = []
    for nb in nbs:
        tok, off = nb.packed_tokens()
        packed.append((torch.from_numpy(np.ascontiguousarray(tok)).cuda(), off))
    with engine.PllScorer(sd, cfg, max_chunk_tokens=8192) as sc:
        alone = []
        for tok, off in packed:
            alone.append(sc.score_device(tok, off).clone())
            torch.cuda.synchronize()
        torch.cuda.synchronize()
        outs = [sc.score_device(tok, off) for tok, off in packed]      # no sync in between
        torch.cuda.synchronize()
        for a, b in zip(alone, outs):
            assert torch.equal(a, b)


def test_degenerate_batches():
    """No hypotheses, only empty hypotheses, a single one-token hypothesis, and stage 4 with N = 0."""
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 6)
    with engine.PllScorer(sd, cfg) as sc:
        assert sc.score_packed(np.zeros(0, np.int32), np.zeros(1, np.int64)).shape == (0,)
        out = sc.score_packed(np.zeros(0, np.int32), np.zeros(4, np.int64))
        assert out.tolist() == [0.0, 0.0, 0.0]
        one, terms = sc.score_packed(np.array([700], np.int32), np.array([0, 1], np.int64), return_token_logp=True)
        exp = pll_oracle.score_hyps(sd, cfg, {"u": {"hyp_1": [700]}})["u"]["hyp_1"]
        assert abs(one[0] - exp) <= PLL_TOL and abs(float(terms[0]) - one[0]) < 1e-6
        mixed = sc.score_packed(np.array([700], np.int32), np.array([0, 0, 1, 1], np.int64))
        assert mixed[0] == 0.0 and mixed[2] == 0.0 and mixed[1] == one[0]
        assert sc.score_cls_packed(np.zeros(0, np.int32), np.zeros(1, np.int64), np.zeros(cfg["hidden"], np.float32), 0.0).shape == (0,)
    assert engine.levenshtein([], []).shape == (0,)
    assert engine.levenshtein([""], [""]).tolist() == [0]
    assert engine.levenshtein(["abc"], [""]).tolist() == [3]


def test_layer0_sharing_is_bit_identical(monkeypatch):
    """Embeddings + the layer-0 Q/K/V projection run on the unique rows of a hypothesis (2L+2)
    instead of on every packed row (L(L+2)); scores, per-token terms and hidden states must be
    bit-identical to the per-copy path, incl. long sequences (streaming attention), chunks that
    fall back (only 1-token hypotheses) and chunk boundaries."""
    cfg = synth.BERT_TINY
    sd = synth.random_init_state_dict(cfg, 8)
    rng = np.random.default_rng(12)
    lens = [1] * 40 + [int(x) for x in rng.integers(1, 40, 150)] + [45, 60, 2, 3, 0, 33, 31, 32]
    toks = [rng.integers(670, 7000, L).astype(np.int32) for L in lens]
    off = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    tok = np.concatenate(toks).astype(np.int32)
    res = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("PLLB_SHARE_L0", mode)
        with engine.PllScorer(sd, cfg, max_chunk_tokens=4096) as sc:
            pll, terms = sc.score_packed(tok, off, return_token_logp=True)
            flops = sc.stats()["gemm_flops"]
        with engine.PllScorer(sd, cfg) as sc:
            h0 = sc.hidden(tok[off[40]:off[60]], off[40:61] - off[40], 0)
            h1 = sc.hidden(tok[off[40]:off[60]], off[40:61] - off[40], 1)
        res[mode] = (pll, terms, h0, h1, flops)
    for a, b in zip(res["1"][:4], res["0"][:4]):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    assert res["1"][4] < res["0"][4]                      # and it executed fewer GEMM FLOPs


# ----------------------------------------------------------------------------- operand types
def test_gemm_fp16_operands_vs_fp32_torch():
    """kind::f16 with IEEE-half operands against a plain fp32 torch matmul of the same (exactly
    representable) operands.  (A = bf16 with W = fp16 is not a usable combination: the descriptor
    has separate format fields, but B200 answers "illegal instruction" — measured in round 2.)"""
    import torch
    torch.manual_seed(5)
    M, N, K = 300, 768, 768
    A = torch.randn(M, K, device="cuda").to(torch.float16)
    W = (torch.randn(N, K, device="cuda") * 0.05).to(torch.float16)
    b = torch.randn(N, device="cuda")
    ref = A.float() @ W.float().T + b
    out32 = engine.debug_gemm(A, W, b, 2, operand_dtype="fp16")
    assert (out32 - ref).abs().max().item() < 1e-3
    out16 = engine.debug_gemm(A, W, b, 0, operand_dtype="fp16")
    assert out16.dtype == torch.float16
    assert ((out16.float() - ref).abs() <= ref.abs() * 2 ** -11 + 1e-3).all()


def test_gelu_epilogue_error_bounds():
    """The bf16-output GELU epilogue is a degree-8 minimax polynomial for erf (no MUFU, FFMA2); the
    fp32-output one is Abramowitz-Stegun 7.1.26.  Bounds over [-6, 6] against erf in float64:
    |err| <= 6e-5 (+ the 16-bit output rounding) and <= 1e-6."""
    import math
    import torch
    M, N, K = 4096, 256, 64
    hi = torch.linspace(-6.0, 6.0, M, device="cuda").bfloat16()
    lo = (torch.linspace(-6.0, 6.0, M, device="cuda") - hi.float()).bfloat16()   # x = hi + lo exactly in fp32
    A = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    A[:, 0], A[:, 1] = hi, lo
    W = torch.zeros(N, K, device="cuda", dtype=torch.bfloat16)
    W[:, 0] = 1.0
    W[:, 1] = 1.0
    b = torch.zeros(N, device="cuda")
    x = (hi.double() + lo.double()).cpu()
    exact = 0.5 * x * (1.0 + torch.tensor([math.erf(v / math.sqrt(2.0)) for v in x.tolist()], dtype=torch.float64))
    out32 = engine.debug_gemm(A, W, b, 3)[:, 0].double().cpu()
    assert (out32 - exact).abs().max().item() <= 1e-6
    for mode, ulp in (("bf16", 2 ** -8), ("fp16", 2 ** -11)):
        a = A if mode == "bf16" else A.to(torch.float16)
        w = W if mode == "bf16" else W.to(torch.float16)
        out16 = engine.debug_gemm(a, w, b, 1, operand_dtype=mode)[:, 0].double().cpu()
        assert ((out16 - exact).abs() <= 6e-5 + exact.abs() * ulp).all(), (mode, (out16 - exact).abs().max().item())


def _golden_pll_case(path):
    gold = json.load(open(path))
    lists = gold["tokens"]
    off = np.zeros(len(lists) + 1, np.int64)
    np.cumsum([len(t) for t in lists], out=off[1:])
    tok = np.array([t for l in lists for t in l], np.int32)
    return gold, tok, off, np.array(gold["pll"], np.float64)


def test_config4_24_layers_L64_vs_reference_golden(gold_dir):
    """BASELINE.json configs[3] shape: bert-large-shaped encoder (24 layers, H 1024), 48 hypotheses
    of 8..64 tokens incl. four at the extremes, against the reference's own run_one_epoch
    (tests/golden/c4_pll_golden.json, oracle/make_golden_c2.py --c4).  fp16 operands — what the c4
    workload of bench.py declares — meet the 0.05-nat bound with a wide margin; bf16 with the fp16
    head is measured; plain bf16 does NOT meet the bound at this depth
    and length (weight rounding alone biases a 64-token PLL by ~0.1 nat), which the test records
    instead of hiding."""
    gold, tok, off, ref = _golden_pll_case(os.path.join(gold_dir, "c4_pll_golden.json"))
    L = np.diff(off)
    assert L.max() == 64 and L.min() == 8 and len(L) >= 40 and gold["cfg"]["num_layers"] == 24
    sd = synth.random_init_state_dict(gold["cfg"], gold["seed"])
    err = {}
    extra = [m for m in os.environ.get("PLLB_C4_GOLDEN_MODES", "").split(",") if m]   # measured and printed only
    for mode in ["fp16", "bf16+fp16head", "bf16"] + extra:
        with engine.PllScorer(sd, gold["cfg"], operand_dtype=mode, max_chunk_tokens=1 << 16) as sc:
            err[mode] = np.abs(sc.score_packed(tok, off) - ref)
        print(f"c4 golden, {mode}: max |dPLL| {err[mode].max():.4f}, mean {err[mode].mean():.4f}, "
              f"rms/sqrt(L) {np.sqrt(np.mean(err[mode] ** 2 / L)):.5f}")
    assert err["fp16"].max() <= PLL_TOL and err["fp16"].mean() <= 0.01, err["fp16"].max()
    for mode in ("bf16+fp16head", "bf16"):                          # bounded, but outside the 0.05-nat tolerance
        assert err[mode].max() <= 0.25, (mode, err[mode].max())
    assert err["fp16"].mean() < err["bf16+fp16head"].mean() <= err["bf16"].mean() * 1.05


def test_c2_2000_utterances_pll_and_one_best_vs_reference_golden(gold_dir):
    """north_star acceptance at a size where it can be evaluated: the first n_utts >= 2000
    utterances x 10-best of the bench workload (BASELINE.json configs[1]) against the reference's
    own run_one_epoch (tests/golden/c2_pll_golden.npz, oracle/make_golden_c2.py): per-hypothesis
    |dPLL| <= 0.05 nats, rescored 1-best identical on >= 99.9 % of the utterances at the weight the
    reference's find_best_weight picks on its own scores; near-ties are counted separately."""
    import zlib
    g = np.load(os.path.join(gold_dir, "c2_pll_golden.npz"))
    n_utts, n_best, ref = int(g["n_utts"]), int(g["n_best"]), g["pll"]
    assert n_utts >= int(os.environ.get("PLLB_C2_GOLDEN_MIN_UTTS", "2000")) and n_best == 10 and len(ref) == n_utts * n_best
    nb = synth.make_nbest(n_utts, n_best, seed=0)
    tok, off = nb.packed_tokens()
    assert zlib.crc32(tok.tobytes()) == int(g["tok_crc"]) and zlib.crc32(off.tobytes()) == int(g["off_crc"])
    sd = synth.random_init_state_dict(synth.BERT_BASE_CHINESE, 10)
    c = rescore_oracle.config(n_best)
    lm_ref = ref.reshape(n_utts, n_best)
    lens = np.array(rescore_oracle.hyps_len_of(nb.hyps, n_best), np.int64)
    dist = oracle.levenshtein_strings([r for r in nb.refs for _ in range(n_best)], [h for hs in nb.hyps for h in hs])
    weights = np.arange(0.0, 1.01, 0.01)
    _, es = oracle.rescore_sweep(nb.am, lm_ref, lens, dist.reshape(n_utts, n_best), weights, 0)
    bw = weights[int(np.argmin(es))]                                   # first strictly smallest CER (rescore.py:41-43)
    s_ref = rescore_oracle.rescore(bw, lens, nb.am, lm_ref, c)
    a_ref = np.argmax(s_ref, -1)
    top2 = np.sort(s_ref, -1)[:, -2:]
    near_tie = (top2[:, 1] - top2[:, 0]) < 0.05 / lens.max()           # a 0.05-nat PLL change could flip these
    modes = os.environ.get("PLLB_C2_GOLDEN_MODES", "bf16,bf16+fp16head,bf16+fp16tail,fp16").split(",")
    for mode in modes:
        with engine.PllScorer(sd, synth.BERT_BASE_CHINESE, operand_dtype=mode) as sc:
            got = sc.score_packed(tok, off)
        err = np.abs(got - ref)
        a_got = np.argmax(rescore_oracle.rescore(bw, lens, nb.am, got.reshape(n_utts, n_best), c), -1)
        same = float((a_got == a_ref).mean())
        _, es_g = oracle.rescore_sweep(nb.am, got.reshape(n_utts, n_best), lens, dist.reshape(n_utts, n_best), weights, 0)
        print(f"c2 golden ({n_utts} utts, weight {bw:.2f}), {mode}: max |dPLL| {err.max():.4f}, mean {err.mean():.4f}, "
              f"> 0.05: {int((err > PLL_TOL).sum())} of {len(err)}; 1-best identical {same:.5f} "
              f"({int((a_got != a_ref).sum())} differ, {int(near_tie.sum())} near-ties); "
              f"edit sum at that weight {int(es_g[int(np.argmin(es))])} vs {int(es.min())}")
        assert same >= 0.999, (mode, same)
        assert (a_got != a_ref)[~near_tie].sum() == 0, "a 1-best changed on an utterance that is not a near-tie"
        if mode in ("bf16", "bf16+fp16head") or (mode.startswith("fp16from:") and int(mode.split(":")[1]) > 6):
            # bf16 operands in (nearly) every encoder layer: sigma(dPLL) ~ 0.003 * sqrt(L), so 0.05 is a 3-4
            # sigma event for the longest hypotheses — rare exceedances are expected at this scale
            # (measured over the whole list: 24 and 2 of 71 760) and are counted, not hidden
            assert err.max() <= 0.08 and np.mean(err <= PLL_TOL) >= 0.9995, (err.max(), int((err > PLL_TOL).sum()))
        else:
            assert err.max() <= PLL_TOL, (mode, err.max())


def test_fp16_conversions_saturate_instead_of_overflowing():
    """One FFN unit driven to 1e5 (> 65504, the largest finite fp16): with fp16 operands the GELU
    output saturates (cvt.rn.satfinite) and every score stays finite; with a bf16 encoder (fp32
    exponent range for activations) the scores still match the fp32 oracle.  Also LayerNorm
    gains scaled 30x (large-magnitude activations) in fp16 mode against the oracle."""
    cfg = synth.BERT_TINY
    nb = synth.make_nbest(6, 3, seed=9)
    tok, off = nb.packed_tokens(cfg["vocab"])
    hyps = {"u": {f"hyp_{i + 1}": [int(t) for t in tok[off[i]:off[i + 1]]] for i in range(len(off) - 1)}}
    sd = synth.random_init_state_dict(cfg, 21, perturb=True)
    sd["bert.encoder.layer.0.intermediate.dense.bias"][7] = 1.0e5
    ref = pll_oracle.score_hyps(sd, cfg, hyps)
    exp = np.array([ref["u"][h] for h in hyps["u"]])
    for mode in ("fp16", "bf16+fp16head", "bf16"):
        with engine.PllScorer(sd, cfg, operand_dtype=mode) as sc:
            got = sc.score_packed(tok, off)
        assert np.isfinite(got).all(), mode
        if mode != "fp16":
            assert np.abs(got - exp).max() <= PLL_TOL, (mode, np.abs(got - exp).max())
    sd = synth.random_init_state_dict(cfg, 21, perturb=True)
    for k in sd:
        if k.startswith("bert.") and k.endswith("LayerNorm.weight"):
            sd[k] = sd[k] * 30.0
    ref = pll_oracle.score_hyps(sd, cfg, hyps)
    exp = np.array([ref["u"][h] for h in hyps["u"]])
    for mode, tol in (("fp16", 0.02), ("bf16+fp16head", PLL_TOL), ("bf16", PLL_TOL)):
        with engine.PllScorer(sd, cfg, operand_dtype=mode) as sc:
            got = sc.score_packed(tok, off)
        assert np.isfinite(got).all() and np.abs(got - exp).max() <= tol, (mode, np.abs(got - exp).max())


def test_two_gpu_drop_in_outputs_identical_to_one_gpu():
    """N GPUs == 1 GPU, bitwise: MLM_PLL/main.py on text and on row-list inputs (num_of_data cutting a
    hypothesis), and rescore.py with the sharded sweep + all_reduce of the CER counts
    (tools/e2e_dropin.py --gpus 2).  Needs two visible B200s; the single-GPU test box skips it, the
    builder's 2-GPU run is kept as profiles/r02_identity_2gpu.log."""
    import subprocess
    import sys
    from asr_rescoring_b200 import _lib
    if _lib.load().pllb_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "e2e_dropin.py"), "--gpus", "2"],
                         capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, (out.stdout + out.stderr)[-3000:]
    assert "identical to the 1-GPU files" in out.stdout and "row-list input" in out.stdout and "sharded sweep" in out.stdout


def test_paired_layernorm_clusters_match_the_single_cta_form(monkeypatch):
    """gemm_ln_kernel<.., PAIR>: cta_group::2 pairs inside the LayerNorm cluster (256-row blocks, M = 256
    MMAs, half of the W box per CTA) against the single-CTA form (PLLB_LN_PAIR=0) and the forced form
    for every launch (PLLB_LN_PAIR=2), for all four cluster sizes and row counts around the 256-row
    block size; and both against the fp32 oracle."""
    rng = np.random.default_rng(7)
    for hidden in (256, 512, 768, 1024):
        cfg = dict(num_layers=3, hidden=hidden, num_heads=hidden // 64, intermediate=4 * hidden, vocab=1300,
                   max_position=64, type_vocab=2, ln_eps=1e-12)
        sd = synth.random_init_state_dict(cfg, 23, perturb=True)
        lens = [int(x) for x in rng.integers(1, 30, size=50)]
        off = np.zeros(len(lens) + 1, np.int64)
        np.cumsum(lens, out=off[1:])
        tok = rng.integers(104, cfg["vocab"], size=int(off[-1])).astype(np.int32)
        got = {}
        for policy in ("0", "1", "2"):
            monkeypatch.setenv("PLLB_LN_PAIR", policy)
            with engine.PllScorer(sd, cfg, max_chunk_tokens=8192) as sc:
                got[policy] = sc.score_packed(tok, off)
        monkeypatch.delenv("PLLB_LN_PAIR", raising=False)
        d1, d2 = np.abs(got["1"] - got["0"]).max(), np.abs(got["2"] - got["0"]).max()
        print(f"H={hidden}: paired vs single-CTA LayerNorm clusters: max |dPLL| default policy {d1:.2e}, forced {d2:.2e}")
        assert d1 <= 2e-3 and d2 <= 2e-3, (hidden, d1, d2)
        hyps = {"u": {f"hyp_{i + 1}": [int(t) for t in tok[off[i]:off[i + 1]]] for i in range(10)}}
        ref = pll_oracle.score_hyps(sd, cfg, hyps)
        for policy in ("0", "2"):
            for i in range(10):
                assert abs(got[policy][i] - ref["u"][f"hyp_{i + 1}"]) <= PLL_TOL, (hidden, policy, i)
