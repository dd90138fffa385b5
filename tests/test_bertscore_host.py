"""Host-side pieces of BERTScore MBR (RMBR): the oracle's greedy matching, the k sweep, the pair
deduplication and blocking of BertScoreFunction, and loud failure without a GPU."""
import numpy as np
import pytest
import torch

from oracle import bertscore_oracle as bo
from asr_rescoring_b200 import _lib, synth
from asr_rescoring_b200.RMBR import mbr
from asr_rescoring_b200.RMBR.utility_functions import BertScoreFunction, dedup_pairs, plan_blocks


def _unit(*v):
    v = torch.tensor(v, dtype=torch.float32)
    return v / v.norm()


def test_greedy_cos_idf_hand_built():
    # reference: [CLS] x1 x2 [SEP]; candidate: [CLS] y1 [SEP].  Only x1, x2 count for recall, every
    # candidate row (incl. its [CLS] / [SEP]) takes part in the max.
    cls, sep = _unit(0, 0, 1), _unit(0, 1, 0)
    x1, x2 = _unit(1, 0, 0), _unit(1, 1, 0)
    y1 = _unit(1, 0, 1)
    ref = torch.stack([cls, x1, x2, sep])
    cand = torch.stack([cls, y1, sep])
    Er, mr, ir = bo.pad_batch([ref])
    Ec, mc, ic = bo.pad_batch([cand])
    P, R, _ = bo.greedy_cos_idf(Er, mr, ir, Ec, mc, ic)
    exp_r = (max(x1 @ cls, x1 @ y1, x1 @ sep) + max(x2 @ cls, x2 @ y1, x2 @ sep)) / 2
    assert abs(float(R[0]) - float(exp_r)) < 1e-6
    exp_p = (max(y1 @ x1, y1 @ x2, y1 @ cls, y1 @ sep))       # precision: candidate interior rows
    assert abs(float(P[0]) - float(exp_p)) < 1e-6
    assert bo.recall_pairs([ref, cand], [1], [0])[0] == pytest.approx(float(exp_r), abs=1e-6)
    # an empty sentence on either side gives exactly 0
    empty = torch.stack([cls, sep])
    assert bo.recall_pairs([ref, empty], [1, 0], [0, 1]).tolist() == [0.0, 0.0]


def test_padding_quirk_negative_cosines():
    """bert_score multiplies the similarity matrix by the padding mask: in a padded batch a reference
    row whose real cosines are all negative gets max 0; scored alone (the contract) it gets the
    true (negative) maximum."""
    cls, sep = _unit(0, 0, 1), _unit(0, 1, 0)
    x = _unit(-1, -0.1, -0.1)
    ref = torch.stack([cls, x, sep])
    short = torch.stack([cls, _unit(1, 0, 0.05), sep])
    long = torch.stack([cls, _unit(1, 0, 0.1), _unit(1, 0.1, 0), sep])
    alone = bo.recall_pairs([ref, short], [1], [0])[0]
    assert alone < 0
    Er, mr, ir = bo.pad_batch([ref, ref])
    Ec, mc, ic = bo.pad_batch([short, long])        # `short` is padded to 4 rows
    R = bo.greedy_cos_idf(Er, mr, ir, Ec, mc, ic)[1]
    assert float(R[0]) == 0.0 and alone == pytest.approx(float(max(x @ cls, x @ short[1], x @ sep)), abs=1e-6)


class _TableUtility:
    """score(cands, refs) read from a [N, n, n] matrix; hypothesis strings encode (utt, index)."""

    def __init__(self, U):
        self.U = U

    def score(self, cands, refs):
        def key(s):
            u, i = s.split(":")
            return int(u), int(i)
        out = []
        for c, r in zip(cands, refs):
            (u, i), (u2, j) = key(c), key(r)
            assert u == u2
            out.append(float(self.U[u, i, j]))
        return out


def test_k_sweep_equals_mbr_decode_per_k():
    rng = np.random.default_rng(4)
    N, n = 40, 10
    U = rng.uniform(0.2, 1.0, size=(N, n, n)).astype(np.float32)
    hyps = [[f"{u}:{i}" for i in range(n)] for u in range(N)]
    util = _TableUtility(U)
    choices = mbr.mbr_choices(U)
    assert sorted(choices) == list(range(2, n + 1))
    for k in range(2, n + 1):
        pred, scores = bo.mbr_decode(k, hyps, util)
        assert [hyps[u][int(i)] for u, i in enumerate(choices[k])] == pred
        np.testing.assert_allclose(mbr.expected_utility(U, k), scores.numpy(), rtol=0, atol=1e-5)


def test_dedup_maps_pairs_to_unique_stripped_strings():
    cands = ["甲乙", " 甲乙", "丙", "", "丙"]
    refs = ["丙", "丁 ", "甲乙", "丁", " "]
    uniq, c, r = dedup_pairs(cands, refs)
    assert uniq == ["甲乙", "丙", "丁", ""]
    assert [uniq[i] for i in c] == [s.strip() for s in cands]
    assert [uniq[i] for i in r] == [s.strip() for s in refs]
    with pytest.raises(ValueError):
        dedup_pairs(["a"], [])


@pytest.mark.parametrize("max_rows", [1, 7, 20, 35, 10 ** 6])
def test_pair_blocks_cover_every_pair_under_the_row_budget(max_rows):
    rng = np.random.default_rng(max_rows)
    n_seq = 12
    seq_rows = rng.integers(2, 9, size=n_seq)
    cand = rng.integers(0, n_seq, size=60).astype(np.int32)
    ref = rng.integers(0, n_seq, size=60).astype(np.int32)
    seen = 0
    for sl, seqs, lc, lr in plan_blocks(cand, ref, seq_rows, max_rows):
        assert sl.start == seen and sl.stop > sl.start
        seen = sl.stop
        assert len(set(seqs.tolist())) == len(seqs)              # each sequence embedded once per block
        assert np.array_equal(seqs[lc], cand[sl]) and np.array_equal(seqs[lr], ref[sl])
        rows = int(seq_rows[seqs].sum())
        assert rows <= max_rows or sl.stop - sl.start == 1
    assert seen == len(cand)


@pytest.mark.skipif(_lib.load().pllb_device_count() > 0, reason="a GPU is present")
def test_bertscore_calls_fail_loudly_without_gpu():
    from asr_rescoring_b200.tokenizer import SyntheticCharTokenizer
    with pytest.raises(_lib.PllbError):
        BertScoreFunction(synth.random_init_state_dict(synth.BERT_TINY, 1), SyntheticCharTokenizer(), num_layers=2,
                          cfg=synth.BERT_TINY)
    lib = _lib.load()
    assert lib.pllb_embed(None, None, None, 0, 0, None, None) == 1
    assert lib.pllb_bertscore(None, None, None, 0, None, None, 0, None, None) == 1
