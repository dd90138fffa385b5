"""Edit-operation alignment on the CPU: the oracle's backtrace against the reference's own
align.py outputs (tests/golden/levenshtein_meta.json) and the pinned distances, the alignment
invariants, and the U/S/I/D counting over hyp_alignment dicts (DESIGN.md §3.10)."""
import json
import os

import numpy as np
import pytest

import oracle
from oracle import align_oracle
from asr_rescoring_b200.cer_clients import GAP
from asr_rescoring_b200.statistic import error_type_count


@pytest.fixture(scope="module")
def kat(gold_dir):
    z = np.load(os.path.join(gold_dir, "levenshtein_kat.npz"))
    with open(os.path.join(gold_dir, "levenshtein_meta.json")) as f:
        return z, json.load(f)


def _word_symbols(ex):
    ids = {w: i for i, w in enumerate(dict.fromkeys(ex["ref"] + ex["hyp"]))}
    return np.array([ids[w] for w in ex["ref"]], np.int32), np.array([ids[w] for w in ex["hyp"]], np.int32)


def test_oracle_reproduces_the_reference_docstring_ops(kat):
    _, meta = kat
    for ex in meta["docstring_examples"]:             # align.py:13-18, run unmodified
        r, h = _word_symbols(ex)
        ops, counts = align_oracle.align_batch(r, [0, len(r)], h, [0, len(h)], np.zeros(1, np.int32))
        assert list(ops[0]) == ex["ops"]
        assert counts[0, 1:].sum() == ex["distance"]
    assert [e["ops"] for e in meta["docstring_examples"]] == [list("UUUD"), list("UUDS")]


def test_oracle_edits_equal_the_pinned_distances(kat):
    z, _ = kat
    n = len(z["dist"])
    ops, counts = align_oracle.align_batch(z["ref_cp"], z["ref_off"], z["hyp_cp"], z["hyp_off"], np.arange(n, dtype=np.int32))
    assert np.array_equal(counts[:, 1:].sum(axis=1), z["dist"])        # Nbest_Align/cer.json, 7 176 pairs
    assert int(counts[:, 1:].sum()) == 3230
    na, nb = np.diff(z["ref_off"]), np.diff(z["hyp_off"])
    assert np.array_equal(counts[:, 0] + counts[:, 1] + counts[:, 2], na)
    assert np.array_equal(counts[:, 0] + counts[:, 1] + counts[:, 3], nb)


def _replay(ref, hyp, ops):
    """Apply ops to ref; returns the hypothesis they describe (and checks U/S against hyp)."""
    out, i, j = [], 0, 0
    for op in ops:
        if op == "U":
            assert ref[i] == hyp[j]
            out.append(ref[i]); i += 1; j += 1
        elif op == "S":
            assert ref[i] != hyp[j]
            out.append(hyp[j]); i += 1; j += 1
        elif op == "I":
            i += 1
        else:
            out.append(hyp[j]); j += 1
    assert i == len(ref)
    return "".join(out)


def test_replaying_ops_gives_the_hypothesis_and_lengths_are_bounded():
    rng = np.random.default_rng(7)
    refs, hyps = [], []
    for _ in range(400):
        alpha = "ab" if rng.random() < 0.5 else "abcdefg"
        refs.append("".join(rng.choice(list(alpha), size=int(rng.integers(0, 40)))))
        hyps.append("".join(rng.choice(list(alpha), size=int(rng.integers(0, 40)))))
    refs += ["", "", "abc"]
    hyps += ["", "xy", ""]
    ops, counts = align_oracle.align_strings(refs, hyps)
    dist = oracle.levenshtein_strings(refs, hyps)
    for r, h, o, c, d in zip(refs, hyps, ops, counts, dist):
        assert _replay(r, h, o) == h
        assert max(len(r), len(h)) <= len(o) <= len(r) + len(h)
        assert c[1] + c[2] + c[3] == d
        assert list(c) == [o.count(x) for x in "USID"]
    assert ops[-3:] == ["", "DD", "III"]


def test_tie_rule_prefers_diagonal_then_up_then_left():
    ops, _ = align_oracle.align_strings(["ab", "a", "ba"], ["ba", "b", "ab"])
    # "ab" -> "ba": S S (diagonal) rather than a gap pair; "a" -> "b": S
    assert ops == ["SS", "S", "SS"]
    ops, _ = align_oracle.align_strings(["aab"], ["ab"])
    assert ops == ["IUU"]                                # diagonal first: the second 'a' is matched
    # up and left tie at (3, 3) and diagonal loses: up (I) is taken; left first would give "IUUD"
    ops, _ = align_oracle.align_strings(["aba", "bab"], ["bab", "aba"])
    assert ops == ["DUUI", "DUUI"]


def test_count_alignment_on_hand_built_alignments():
    ali = {
        "utt1": {"hyp_1": [list("ab") + [GAP], list("a") + [GAP] + list("c"), list("UID")],
                 "hyp_2": [list("ab"), list("xb"), list("SU")]},
        "utt2": {"hyp_1": [[GAP], list("z"), ["D"]]},
        "utt3": {"hyp_1": [[], [], []]},
    }
    got = error_type_count.count_alignment(ali)
    assert got["total"] == {"U": 2, "S": 1, "I": 1, "D": 2}
    assert got["per_rank"] == {"hyp_1": {"U": 1, "S": 0, "I": 1, "D": 2}, "hyp_2": {"U": 1, "S": 1, "I": 0, "D": 0}}
    assert error_type_count.count_alignment({}) == {"total": dict.fromkeys("USID", 0), "per_rank": {}}


def test_gap_placement_follows_the_op():
    """An I leaves the hypothesis side empty, a D the reference side; joining a side without the
    gaps gives back its string."""
    ali = {"u": {"hyp_1": [["a", "b", GAP], ["a", GAP, "c"], ["U", "I", "D"]]}}
    ref, hyp, ops = ali["u"]["hyp_1"]
    for r, h, o in zip(ref, hyp, ops):
        assert (h == GAP) == (o == "I") and (r == GAP) == (o == "D")
    assert "".join(ref) == "ab" and "".join(hyp) == "ac"
    assert GAP == ""
