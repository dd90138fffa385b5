"""Edit-operation alignment on the B200 (align_kernel, pllb_align / pllb_align_host): bit-exact
against the C restatement of the backtrace (oracle/align_oracle.c), consistent with the Levenshtein
kernel, and end to end through cer_clients.hyp_alignment and statistic.error_type_count."""
import ctypes
import json
import os

import numpy as np
import pytest

from oracle import align_oracle, rescore_oracle
from asr_rescoring_b200 import _lib, cer_clients, engine, synth
from asr_rescoring_b200.statistic import error_type_count

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("require_gpu")]

LENGTHS = [0, 1, 31, 32, 33, 63, 64, 65, 128, 513, 1024]


def _check_against_oracle(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref):
    al = engine.align_packed(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref)
    ops_o, counts_o = align_oracle.align_batch(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref)
    got = [al.op_string(i) for i in range(len(al))]
    assert got == ops_o
    assert np.array_equal(al.n_ops, [len(o) for o in ops_o])
    assert np.array_equal(al.counts, counts_o)
    # counts are a bincount of the ops; S + I + D is the Levenshtein kernel's distance
    for i in range(len(al)):
        assert np.array_equal(al.counts[i], [np.count_nonzero(al[i] == ord(c)) for c in "USID"])
    dist = engine.levenshtein_packed(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref)
    assert np.array_equal(al.counts[:, 1:].sum(axis=1), dist)
    # the slot past the ops is zero
    for i in range(len(al)):
        assert not al.ops[int(al.off[i]) + int(al.n_ops[i]):int(al.off[i + 1])].any()
    return al


def test_reference_kats_and_docstring_examples_bit_exact(gold_dir):
    z = np.load(os.path.join(gold_dir, "levenshtein_kat.npz"))
    n = len(z["dist"])
    al = _check_against_oracle(z["ref_cp"], z["ref_off"], z["hyp_cp"], z["hyp_off"], np.arange(n, dtype=np.int32))
    assert np.array_equal(al.counts[:, 1:].sum(axis=1), z["dist"]) and int(al.counts[:, 1:].sum()) == 3230
    with open(os.path.join(gold_dir, "levenshtein_meta.json")) as f:
        meta = json.load(f)
    for ex in meta["docstring_examples"]:                 # align.py:13-18, words as opaque symbols
        ids = {w: i for i, w in enumerate(dict.fromkeys(ex["ref"] + ex["hyp"]))}
        r = np.array([ids[w] for w in ex["ref"]], np.int32)
        h = np.array([ids[w] for w in ex["hyp"]], np.int32)
        a = engine.align_packed(r, [0, len(r)], h, [0, len(h)], np.zeros(1, np.int32))
        assert list(a.op_string(0)) == ex["ops"]
    assert engine.align(["你好嗎"], [" 你好不好 "]).op_string(0) == "UUDS"


def test_config1_shape_bit_exact():
    nb = synth.make_nbest(100, 10, seed=1)
    refs = [r.strip() for r in nb.refs]
    hyps = [h.strip() for hs in nb.hyps for h in hs]
    rc, ro = engine.pack_strings(refs)
    hc, ho = engine.pack_strings(hyps)
    _check_against_oracle(rc, ro, hc, ho, np.repeat(np.arange(len(refs), dtype=np.int32), 10))


def _binary_pairs(seed, lengths, per=2):
    rng = np.random.default_rng(seed)
    refs, hyps = [], []
    for la in lengths:
        for lb in lengths:
            for _ in range(per):
                refs.append(rng.integers(0, 2, size=la).astype(np.int32))
                hyps.append(rng.integers(0, 2, size=lb).astype(np.int32))
    pack = lambda xs: (np.concatenate(xs + [np.zeros(0, np.int32)]),
                       np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.int64))
    return pack(refs) + pack(hyps)


@pytest.mark.parametrize("lengths", [LENGTHS, [0, 1, 31, 32, 33, 63, 64], [0, 1, 63, 64, 65, 128]])
def test_two_symbol_alphabet_ties_at_block_edges(lengths):
    """Two symbols force ties nearly everywhere.  The full list mixes shared-memory and global
    code slots in one launch; the shorter lists run the shared-memory-only and mid-width launches."""
    rc, ro, hc, ho = _binary_pairs(len(lengths), lengths)
    _check_against_oracle(rc, ro, hc, ho, np.arange(len(ro) - 1, dtype=np.int32))


def _dev(a, torch):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_device_entry_equals_host_entry_and_runs_repeat_bit_exactly():
    import torch
    rc, ro, hc, ho = _binary_pairs(5, [0, 3, 40, 64, 65, 300])
    n = len(ho) - 1
    pair_ref = np.arange(n, dtype=np.int32)
    host = engine.align_packed(rc, ro, hc, ho, pair_ref)
    again = engine.align_packed(rc, ro, hc, ho, pair_ref)
    assert np.array_equal(host.ops, again.ops) and np.array_equal(host.n_ops, again.n_ops)
    assert np.array_equal(host.counts, again.counts)
    lib = _lib.load()
    t = [_dev(x, torch) for x in (rc, ro, hc, ho, pair_ref, host.off)]
    ops = torch.full((len(host.ops),), 0xAB, dtype=torch.uint8, device="cuda")
    n_ops = torch.zeros(n, dtype=torch.int32, device="cuda")
    counts = torch.zeros((n, 4), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pllb_align(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), n,
                              300, t[5].data_ptr(), ops.data_ptr(), n_ops.data_ptr(), counts.data_ptr(), stream))
    torch.cuda.synchronize()
    assert np.array_equal(ops.cpu().numpy(), host.ops)
    assert np.array_equal(n_ops.cpu().numpy(), host.n_ops) and np.array_equal(counts.cpu().numpy(), host.counts)
    # a pair longer than the max_len the launch was sized for is flagged, not aligned
    n_ops.zero_()
    _lib.check(lib.pllb_align(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), n,
                              64, t[5].data_ptr(), ops.data_ptr(), n_ops.data_ptr(), counts.data_ptr(), stream))
    torch.cuda.synchronize()
    na = np.diff(ro)
    nb = np.diff(ho)
    too_long = (na > 64) | (nb > 64)
    got = n_ops.cpu().numpy()
    assert (got[too_long] == -1).all() and np.array_equal(got[~too_long], host.n_ops[~too_long])
    assert not counts.cpu().numpy()[too_long].any()


def test_rejections():
    with pytest.raises(_lib.PllbError) as e:
        engine.align(["a"], ["b" * 1025])
    assert e.value.code == 5                              # PLLB_ERR_TOO_LONG, hypothesis side
    with pytest.raises(_lib.PllbError) as e:
        engine.align(["a" * 1025], ["b"])
    assert e.value.code == 5                              # reference side
    with pytest.raises(_lib.PllbError) as e:
        engine.align(["ab"], ["ab", "cd"], pair_ref=[0, 1])
    assert e.value.code == 1                              # pair_ref out of range
    with pytest.raises(_lib.PllbError) as e:
        engine.align(["ab"], ["ab"], pair_ref=[-1])
    assert e.value.code == 1
    cp = np.arange(6, dtype=np.int32)
    with pytest.raises(_lib.PllbError) as e:             # hypothesis offsets not ascending
        engine.align_packed(cp, [0, 3], cp, [0, 4, 2], np.zeros(2, np.int32))
    assert e.value.code == 1
    with pytest.raises(_lib.PllbError) as e:             # reference offsets not ascending
        engine.align_packed(cp, [0, 4, 2], cp, [0, 2], np.zeros(1, np.int32))
    assert e.value.code == 1
    lib = _lib.load()
    n_ops = np.zeros(1, np.int32)
    counts = np.zeros(4, np.int32)
    ops = np.zeros(8, np.uint8)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    ro, ho, pr = np.array([0, 3], np.int64), np.array([0, 3], np.int64), np.zeros(1, np.int32)
    short = np.array([0, 5], np.int64)                    # a slot shorter than na + nb = 6
    assert lib.pllb_align_host(p(cp), p(ro), 1, p(cp), p(ho), p(pr), 1, p(short), p(ops), p(n_ops), p(counts)) == 1


def test_hyp_alignment_end_to_end_and_error_split_of_the_rescored_one_best():
    nb = synth.make_nbest(300, 10, seed=21)
    got = cer_clients.hyp_alignment(nb.hyps_text(), nb.ref_text())
    refs, hyps = [], []
    for u, hs in nb.hyps_text().items():
        for h in hs.values():
            refs.append(nb.ref_text()[u].strip())
            hyps.append(h.strip())
    ops_o, _ = align_oracle.align_strings(refs, hyps)
    want, p = {}, 0
    for u, hs in nb.hyps_text().items():
        want[u] = {}
        for k in hs:
            r, h, o = refs[p], hyps[p], ops_o[p]
            ar, ah, i, j = [], [], 0, 0
            for op in o:
                ar.append(cer_clients.GAP if op == "D" else r[i])
                ah.append(cer_clients.GAP if op == "I" else h[j])
                i += op != "D"
                j += op != "I"
            want[u][k] = [ar, ah, list(o)]
            p += 1
    assert got == want
    tot = error_type_count.count_alignment(got)["total"]
    assert tot["S"] + tot["I"] + tot["D"] == int(engine.levenshtein(refs, hyps).sum())

    from asr_rescoring_b200 import rescore as dropin
    lm = synth.synthetic_lm_scores(nb, seed=6)
    cfg = rescore_oracle.config(10)
    bw, bc = dropin.find_best_weight(nb.am.tolist(), lm.tolist(), nb.hyps, nb.refs, cfg)
    s = dropin.rescore(bw, dropin._hyps_len(nb.hyps, 10), nb.am.tolist(), lm.tolist(), cfg)
    best = dropin.get_highest_score_hyp(s, nb.hyps)
    c = error_type_count.error_counts(nb.refs, best)
    assert c["S"] + c["I"] + c["D"] == round(bc * sum(len(r.strip()) for r in nb.refs))
    assert c["U"] + c["S"] + c["I"] == sum(len(r.strip()) for r in nb.refs)
