"""Host-side logic (CPU): synthetic data, config/CLI surface, tokenizer, sharding and the
world-size-2 gloo path of the score gather / count reduce."""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from asr_rescoring_b200 import shard, synth
from asr_rescoring_b200.tokenizer import BertCharTokenizer, SyntheticCharTokenizer
from asr_rescoring_b200.util.arg_parser import ArgParser
from asr_rescoring_b200.util.config import parse_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_synth_is_deterministic_and_aishell_shaped():
    a, b = synth.make_nbest(50, 10, seed=0), synth.make_nbest(50, 10, seed=0)
    assert a.hyps == b.hyps and np.array_equal(a.am, b.am)
    assert (np.diff(a.am, axis=1) <= 0).all()              # AM scores sorted descending
    assert all(len(h) >= 1 for hs in a.hyps for h in hs)
    tok, off = a.packed_tokens()
    assert tok.min() >= 670 and tok.max() < 670 + 7322 and len(off) == 501
    ref_len, edits = synth.shape_table()                   # espnet_data/alfred/test/{ref_text,hyps_cer}.json
    assert len(ref_len) == 7176 and int(ref_len.sum()) == 104765 and int(edits.sum()) == 118889
    hist = dict(zip(*np.unique(ref_len, return_counts=True)))
    assert hist == synth.REF_LEN_HIST
    assert dict(zip(*np.unique(edits, return_counts=True))) == synth.EDIT_HIST
    assert [len(r) for r in a.refs] == list(ref_len[:50]) and np.array_equal(a.edits, edits[:50])


def test_random_init_keys_match_hf_state_dict_names():
    sd = synth.random_init_state_dict(synth.BERT_TINY, 3)
    assert sd["cls.predictions.decoder.weight"] is sd["bert.embeddings.word_embeddings.weight"]
    assert float(sd["bert.embeddings.word_embeddings.weight"][0].abs().sum()) == 0.0
    assert synth.config_from_state_dict(sd)["num_layers"] == 2
    try:
        from transformers import BertConfig, BertForMaskedLM
    except Exception:
        pytest.skip("transformers not importable")
    c = synth.BERT_TINY
    hf = BertForMaskedLM(BertConfig(vocab_size=c["vocab"], hidden_size=c["hidden"], num_hidden_layers=c["num_layers"],
                                    num_attention_heads=c["num_heads"], intermediate_size=c["intermediate"],
                                    max_position_embeddings=c["max_position"]))
    hf_keys = {k for k in hf.state_dict() if "position_ids" not in k}
    assert hf_keys == set(sd.keys())


def test_config_surface(tmp_path):
    p = tmp_path / "c.yaml"
    p.write_text(open(os.path.join(ROOT, "asr-rescoring_b200", "MLM_PLL", "config", "score.yaml")).read())
    cfg = ArgParser().parse(["--config", str(p)])
    assert cfg.task == "scoring" and cfg.seed == 10 and cfg.dataloader.batch_size == 32 and cfg.model.bert == "bert-base-chinese"
    with pytest.raises(AttributeError):     # the reference's only error convention
        _ = cfg.missing_key
    assert parse_config({"a": {"b": 1}}).a.b == 1
    with pytest.raises(SystemExit):
        ArgParser().parse([])


def test_tokenizer_matches_transformers_bert_tokenizer(tmp_path):
    vocab = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", "你", "好", "嗎", "a", "ab", "##c", "##d", "hello", "1", "##2", ",", "。"]
    vp = tmp_path / "vocab.txt"
    vp.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    mine = BertCharTokenizer(str(vp))
    texts = ["你好嗎", "你好 abc Hello,12。", "未知字 abcd xyz", "  你  好 ", "ABD", ""]
    try:
        from transformers import BertTokenizer
        hf = BertTokenizer(str(vp))
    except Exception:
        hf = None
    for t in texts:
        toks = mine.tokenize(t)
        if hf is not None:
            assert toks == hf.tokenize(t), t
            assert mine.convert_tokens_to_ids(toks) == hf.convert_tokens_to_ids(toks)
    assert mine.tokenize("你好abc") == ["你", "好", "ab", "##c"]
    assert SyntheticCharTokenizer().encode("你好") == [synth.synthetic_token_id("你"), synth.synthetic_token_id("好")]


def test_lpt_partition_is_balanced_and_deterministic():
    rng = np.random.default_rng(0)
    lens = [[int(x) for x in rng.integers(3, 38, size=10)] for _ in range(500)]
    costs = shard.utterance_costs(lens)
    for world in (1, 2, 4, 8):
        parts = shard.lpt_partition(costs, world)
        allidx = np.sort(np.concatenate(parts))
        assert np.array_equal(allidx, np.arange(500))
        loads = np.array([costs[p].sum() for p in parts])
        assert loads.max() <= loads.mean() * 1.02 + costs.max()
        again = shard.lpt_partition(costs, world)
        assert all(np.array_equal(a, b) for a, b in zip(parts, again))


def test_drop_in_function_surface():
    import importlib
    m = importlib.import_module("asr_rescoring_b200.MLM_PLL.main")
    r = importlib.import_module("asr_rescoring_b200.rescore")
    for name in ("MyDataset", "collate", "set_dataloader", "run_one_epoch", "pll_bert_scoring", "mlm_finetune_bert"):
        assert hasattr(m, name)
    for name in ("dict_to_list", "find_best_weight", "rescore", "get_highest_score_hyp", "cer"):
        assert hasattr(r, name)
    assert r.dict_to_list({"u1": {"hyp_1": 1.0, "hyp_2": 2.0}, "u2": "abc"}) == [[1.0, 2.0], "abc"]
    assert r.get_highest_score_hyp(np.array([[0.1, 0.3, 0.3], [np.nan, 1.0, 2.0]]), [["a", "b", "c"], ["d", "e", "f"]]) == ["b", "d"]
    rows = [{"utt_id": "u", "hyp_id": "hyp_1"}, {"utt_id": "u", "hyp_id": "hyp_2"}, {"utt_id": "v", "hyp_id": "hyp_1"}]
    assert m.skeleton_from_rows(rows) == {"u": {"hyp_1": 0, "hyp_2": 0}, "v": {"hyp_1": 0}}
    with pytest.raises(KeyError):            # quirk 3: no hyp_1 row for an utterance
        m.skeleton_from_rows([{"utt_id": "w", "hyp_id": "hyp_2"}])
    with pytest.raises(TypeError):                # train_mode needs a trainer, with or without do_scoring
        m.run_one_epoch(None, object(), [], {}, train_mode=True, do_scoring=True)
    with pytest.raises(TypeError):                # the loss / training pass needs a trainer, not a scorer
        m.run_one_epoch(None, object(), [], None, train_mode=True, do_scoring=False)


def test_preprocess_rows_match_reference_schema():
    import importlib
    p = importlib.import_module("asr_rescoring_b200.MLM_PLL.preprocess")
    from oracle import pll_oracle
    tk = SyntheticCharTokenizer()
    rows = p.do_job("你好嗎", "utt", "hyp_1", "for_scoring", [], tokenizer=tk)
    assert rows == pll_oracle.expand_rows(tk.encode("你好嗎"), "utt", "hyp_1")
    packed = p.pack_hyps_text({"u": {"hyp_1": "你好", "hyp_2": ""}}, tk)
    assert packed["offsets"] == [0, 2, 2] and packed["format"] == "pllb-packed-v1"


GLOO_WORKER = textwrap.dedent("""
    import os, sys, json
    import numpy as np
    sys.path.insert(0, os.environ["PLLB_ROOT"])
    import torch.distributed as dist
    from asr_rescoring_b200 import shard
    rank, world, _ = shard.init_process_group(backend="gloo")
    rng = np.random.default_rng(0)
    lens = [[int(x) for x in rng.integers(1, 30, size=4)] for _ in range(37)]
    parts = shard.lpt_partition(shard.utterance_costs(lens), world)
    base = np.arange(0, 37 * 4 + 1, 4)
    # stand-in per-hypothesis "scores": a deterministic function of the global hypothesis index
    idx = np.array([base[u] + k for u in parts[rank] for k in range(4)], np.int64)
    vals = -np.sqrt(idx.astype(np.float64) + 1.0) * 3.3
    full = shard.gather_scores(vals, idx, 37 * 4)
    counts = shard.reduce_counts(np.array([len(idx), int(idx.sum())], np.int64))
    if rank == 0:
        print(json.dumps({"ok": bool(np.array_equal(full, -np.sqrt(np.arange(148) + 1.0) * 3.3)),
                          "counts": counts.tolist()}))
    dist.destroy_process_group()
""")


GLOO_STRONG_WORKER = textwrap.dedent("""
    import json, os, sys
    import numpy as np
    sys.path.insert(0, os.environ["PLLB_ROOT"])
    import torch.distributed as dist
    from asr_rescoring_b200 import shard, synth
    rank, world, _ = shard.init_process_group("gloo")
    n_best = 5
    nb = synth.make_nbest(41, n_best, seed=3)                 # odd count: ranks own different numbers of hypotheses
    lens = [[len(h) for h in hs] for hs in nb.hyps]
    parts = shard.lpt_partition(shard.utterance_costs(lens), world)
    mine = parts[rank]
    idx = shard.global_hyp_index(mine, n_best)
    score = lambda i: -np.sqrt(i.astype(np.float64) + 1.0) * 1.7     # stands in for the PLL of global hypothesis i
    full = shard.gather_scores(score(idx), idx, 41 * n_best)
    # sharded sweep plumbing of rescore.py: contiguous blocks, integer all_reduce, argmax gather
    lo, hi = shard.block_range(41, rank, world)
    counts = shard.reduce_counts(np.array([hi - lo, sum(len(r) for r in nb.refs[lo:hi])], np.int64))
    arg = shard.gather_blocks(np.arange(lo, hi, dtype=np.int32)[None, :].repeat(3, 0), 41, axis=1)
    if rank == 0:
        print(json.dumps({"ok": bool(np.array_equal(full, score(np.arange(41 * n_best)))),
                          "sizes": [int(len(p)) for p in parts], "counts": counts.tolist(),
                          "arg_ok": bool(np.array_equal(arg, np.arange(41, dtype=np.int32)[None, :].repeat(3, 0))),
                          "ref_len": sum(len(r) for r in nb.refs)}))
    dist.destroy_process_group()
""")


def test_gloo_world_size_2_strong_scaling_partition_and_gather(tmp_path):
    """The N > 1 path of bench.py / MLM_PLL/main.py / rescore.py on CPU: LPT partition with unequal
    per-rank hypothesis counts, global indices, score gather, count reduction, argmax gather."""
    script = tmp_path / "s.py"
    script.write_text(GLOO_STRONG_WORKER)
    env = dict(os.environ, PLLB_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29573", str(script)],
                         env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert res["ok"] and res["arg_ok"] and sum(res["sizes"]) == 41 and res["sizes"][0] != res["sizes"][1]
    assert res["counts"] == [41, res["ref_len"]]


def test_build_is_serialised_by_a_file_lock():
    from asr_rescoring_b200 import build as b
    import inspect
    src = inspect.getsource(b.build) + inspect.getsource(b._build_locked)
    assert "fcntl.flock" in src and "os.replace" in src
    assert b.build() == b.LIB                                  # fresh library: returns without compiling


def test_text_input_refuses_the_synthetic_tokenizer_with_a_real_checkpoint(tmp_path):
    """ADVICE r1: a checkpoint scored with made-up token ids must raise, not write plausible files."""
    import torch
    from types import SimpleNamespace
    from asr_rescoring_b200.MLM_PLL import main as m
    ckpt = tmp_path / "ckpt.pt"
    torch.save({}, ckpt)
    cfg_ckpt = SimpleNamespace(checkpoint_path=str(ckpt), model=SimpleNamespace(bert="bert-base-chinese"))
    with pytest.raises(FileNotFoundError):
        m._tokenizer(cfg_ckpt)
    cfg_none = SimpleNamespace(checkpoint_path="", model=SimpleNamespace(bert="bert-base-chinese"))
    with pytest.raises(FileNotFoundError):
        m._tokenizer(cfg_none)
    cfg_rand = SimpleNamespace(checkpoint_path="", model=SimpleNamespace(bert="bert-base-chinese", random_init_seed=10))
    assert isinstance(m._tokenizer(cfg_rand), SyntheticCharTokenizer)
    packed = tmp_path / "p.json"
    packed.write_text(json.dumps({"format": "pllb-packed-v1", "tokenizer": "synthetic", "utt_id": ["u"], "hyp_id": ["hyp_1"],
                                  "tokens": [700], "offsets": [0, 1]}))
    with pytest.raises(ValueError):
        m.load_split(str(packed), None, cfg_ckpt)
    assert m.load_split(str(packed), None, cfg_rand)[1] == {"u": {"hyp_1": [700]}}


def test_gloo_world_size_2_gather_and_reduce(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, PLLB_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29571", str(script)],
                         env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    assert res["ok"] and res["counts"] == [148, sum(range(148))]


def _table_lookup_reference(table, text):
    """numpy restatement of pllb_tokenize_host for one string: ids, or None if flagged."""
    cps = [ord(c) for c in text]
    t = [int(table[c]) if c < len(table) else -3 for c in cps]
    if any(x == -3 for x in t):
        return None
    return [x for x in t if x >= 0]


def test_char_table_agrees_with_the_wordpiece_tokenizer(tmp_path):
    from asr_rescoring_b200.tokenizer import TOK_REMOVED, TOK_SPACE, TOK_WORD
    vocab = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", "你", "好", "嗎", "豈", "a", "ab", "##c", "1", ",", "。", "，", "!", "$"]
    vp = tmp_path / "vocab.txt"
    vp.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    tk = BertCharTokenizer(str(vp))
    table = tk.char_table()
    assert table[ord("你")] == 5 and table[ord("龘")] == 1            # in vocab / [UNK]
    assert table[0xF900] == vocab.index("豈")                         # compatibility ideograph -> NFC form
    assert table[ord(" ")] == TOK_SPACE and table[0x3000] == TOK_SPACE
    assert table[0] == TOK_REMOVED and table[0xFFFD] == TOK_REMOVED and table[0x200B] == TOK_REMOVED
    assert table[ord("a")] == TOK_WORD and table[ord("1")] == TOK_WORD and table[0x0301] == TOK_WORD
    assert table[ord("あ")] == TOK_WORD                               # kana is not split by BasicTokenizer
    assert table[ord(",")] == vocab.index(",") and table[ord("?")] == 1
    rng = np.random.default_rng(5)
    alphabet = list("你好嗎豈龘，。,!?$ \t\u3000\x00\ufffd\u200b") + [chr(0xF900), chr(0x20000)]
    for _ in range(300):
        text = "".join(rng.choice(alphabet, size=int(rng.integers(0, 12))))
        assert _table_lookup_reference(table, text) == tk.encode(text), repr(text)
    assert _table_lookup_reference(table, "你好abc") is None
    syn = SyntheticCharTokenizer()
    st = syn.char_table()
    for text in ("你好嗎", "abc 1", "龘\u3000x"):
        assert _table_lookup_reference(st, text) == syn.encode(text)


def test_encode_batch_merges_device_and_host_paths(tmp_path, monkeypatch):
    """Host logic of tokenizer.encode_batch with the device call replaced by its numpy restatement:
    flagged hypotheses are re-tokenised on the host and spliced back in order."""
    from asr_rescoring_b200 import engine, tokenizer as tkmod

    def fake_tokenize_packed(table, cp, cp_off):
        ids, off, flag = [], [0], []
        for i in range(len(cp_off) - 1):
            text = "".join(chr(c) for c in cp[cp_off[i]:cp_off[i + 1]])
            r = _table_lookup_reference(table, text)
            flag.append(1 if r is None else 0)
            ids += r or []
            off.append(len(ids))
        return np.array(ids, np.int32), np.array(off, np.int64), np.array(flag, np.uint8)

    monkeypatch.setattr(engine, "tokenize_packed", fake_tokenize_packed)
    vocab = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", "你", "好", "嗎", "a", "ab", "##c", "1", "##2", ",", "。", "hello"]
    vp = tmp_path / "vocab.txt"
    vp.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    tk = BertCharTokenizer(str(vp))
    strings = ["你好", "abc", "", "你 好，嗎", "hello 12", "好", "a你", "。。", "12"]
    for sel in (strings, strings[::-1], ["abc", "12"], ["你好", "嗎"], []):
        ids, off = tkmod.encode_batch(tk, sel)
        assert off.tolist() == np.concatenate([[0], np.cumsum([len(tk.encode(x)) for x in sel])]).astype(int).tolist()
        for i, x in enumerate(sel):
            assert ids[off[i]:off[i + 1]].tolist() == tk.encode(x), x


def test_bench_reference_arm_prints_one_json_line_with_the_contract_keys():
    """bench.py --impl reference runs on the host cores alone (no GPU): exactly one line on
    stdout, carrying the keys the driver reads."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-sample-hyps", "10"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "N-best PLL hypotheses/sec" and d["unit"] == "hyps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    # baseline/_ref (the unmodified reference files, baseline/install_ref.py) is what runs when present
    expect = "reference" if os.path.exists(os.path.join(root, "baseline", "_ref", "MLM_PLL", "main.py")) else "port"
    assert d["cpu_baseline"]["kind"] == expect and d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]


def test_bench_reference_arm_combiner_workload():
    """--workload c5 --impl reference: the reference's find_best_weight on a reduced list."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "c5",
                          "--utts", "40", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert d["impl"] == "reference" and d["value"] > 0 and 0.0 <= d["best_weight"] <= 1.0 and d["dtype"] == "f64"


def test_bench_rejects_zero_steps_and_dump_outputs_of_the_reference_arm():
    import bench
    assert bench.parse_args(["--steps", "2", "--dump-outputs", "d"]).steps == 2
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]):
        with pytest.raises(SystemExit):
            bench.parse_args(argv)


def test_bench_write_outputs_keeps_a_seeded_sample_within_the_limit(tmp_path):
    import bench
    rng = np.random.default_rng(1)
    arrays = {"pll": rng.normal(size=5000), "argmax": rng.integers(0, 10, (101, 300)).astype(np.float32)}
    bench.write_outputs(str(tmp_path / "all"), arrays)
    for name, a in arrays.items():
        assert np.array_equal(np.load(tmp_path / "all" / f"{name}.npy"), a)
    assert sorted(os.listdir(tmp_path / "all")) == ["argmax.npy", "pll.npy"]
    limit = 60000                                       # both arrays (161 200 bytes) over it
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["argmax.npy", "argmax_index.npy", "pll.npy", "pll_index.npy"] == sorted(os.listdir(tmp_path / "b"))
    assert sum(np.load(tmp_path / "a" / f).nbytes for f in files) <= limit
    for name, a in arrays.items():
        idx = np.load(tmp_path / "a" / f"{name}_index.npy")
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype == a.dtype and np.array_equal(got, a[..., idx.astype(np.int64)])
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))
        assert np.all(np.diff(idx) > 0)


def test_pack_stripped_equals_strip_then_pack():
    """The combiner's one-pass packing (raw lengths for rescore.py:28-35, stripped code points for the
    CER) against the plain per-string strip(), incl. every whitespace code point str.strip() knows."""
    from asr_rescoring_b200 import engine
    for strs in (["你好", " a b ", "", "　x　", "xyz\n", "\x85q", " "], ["abc", "", "好"], []):
        cp, off, raw = engine.pack_stripped(strs)
        cp2, off2 = engine.pack_strings([s.strip() for s in strs])
        assert np.array_equal(cp, cp2) and np.array_equal(off, off2) and list(raw) == [len(s) for s in strs]
    assert sorted(c for c in range(0x110000) if chr(c).isspace()) == sorted(engine._whitespace_code_points().tolist())


def test_preprocess_main_writes_the_three_packed_splits(tmp_path):
    """MLM_PLL/preprocess.py __main__ (reference: preprocess.py:33-72): the three for_scoring jobs, run
    from an MLM_PLL working directory with the relative paths of the reference."""
    tk = SyntheticCharTokenizer()
    (tmp_path / "MLM_PLL").mkdir()
    texts = {}
    for split in ("train", "dev", "test"):
        d = tmp_path / "espnet_data" / "alfred" / split
        d.mkdir(parents=True)
        texts[split] = {f"{split}_u{i}": {"hyp_1": "你好嗎", "hyp_2": "", "hyp_3": "好"} for i in range(3)}
        (d / "hyps_text.json").write_text(json.dumps(texts[split], ensure_ascii=False), encoding="utf-8")
        (d / "ref_text.json").write_text(json.dumps({f"{split}_u{i}": "你好" for i in range(2)}, ensure_ascii=False),
                                         encoding="utf-8")
    script = os.path.join(ROOT, "asr-rescoring_b200", "MLM_PLL", "preprocess.py")
    env = {k: v for k, v in os.environ.items() if k != "PLLB_VOCAB"}
    out = subprocess.run([sys.executable, script], cwd=tmp_path / "MLM_PLL", env=env, capture_output=True, text=True)
    assert out.returncode != 0 and "PLLB_VOCAB" in (out.stderr + out.stdout)        # no silent synthetic tokenizer
    out = subprocess.run([sys.executable, script], cwd=tmp_path / "MLM_PLL", env=dict(env, PLLB_SYNTHETIC_TOKENIZER="1"),
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-1500:]
    for split in ("train", "dev", "test"):
        p = json.load(open(tmp_path / "MLM_PLL" / "preprocessed_data" / "for_scoring" / f"{split}.json", encoding="utf-8"))
        assert p["format"] == "pllb-packed-v1" and p["tokenizer"] == "synthetic"
        assert p["utt_id"] == [u for u in texts[split] for _ in range(3)] and p["hyp_id"] == ["hyp_1", "hyp_2", "hyp_3"] * 3
        assert p["offsets"] == [0, 3, 3, 4, 7, 7, 8, 11, 11, 12] and p["tokens"][:3] == tk.encode("你好嗎")
    from oracle import pll_oracle
    for split in ("train", "dev"):                    # the two for_training jobs: the reference's row list
        rows = json.load(open(tmp_path / "MLM_PLL" / "preprocessed_data" / "for_training" / f"{split}.json", encoding="utf-8"))
        exp = [r for i in range(2) for r in pll_oracle.expand_rows(tk.encode("你好"), f"{split}_u{i}", None)]
        assert rows == exp


def test_training_batches_match_collate_and_dataloader_order():
    from types import SimpleNamespace
    """pad_batch == the reference's collate (MLM_PLL/main.py:28-54, via the oracle restatement);
    RowLoader(shuffle=True) yields the order torch's DataLoader yields under the same global seed
    (MLM_PLL/main.py:57-70 with config.shuffle)."""
    import importlib
    import torch
    from torch.utils.data import DataLoader
    from oracle import pll_oracle, train_oracle
    m = importlib.import_module("asr_rescoring_b200.MLM_PLL.main")
    rows = train_oracle.training_rows([[200, 201, 202], [300], [400, 401, 402, 403, 404], [500, 501]])
    ids, am, lab = m.pad_batch(rows[:7])
    o_ids, o_am, o_lab, *_ = pll_oracle.collate(rows[:7])
    assert np.array_equal(ids, o_ids.numpy()) and np.array_equal(am, o_am.numpy()) and np.array_equal(lab, o_lab.numpy())
    conf = SimpleNamespace(shuffle=True, batch_size=3, num_worker=0)
    torch.manual_seed(10)
    mine = [[r["input_ids"] for r in b] for b in m.set_dataloader(conf, m.MyDataset(rows), False)]
    mine += [[r["input_ids"] for r in b] for b in m.set_dataloader(conf, m.MyDataset(rows), False)]    # a second epoch
    torch.manual_seed(10)
    dl = DataLoader(dataset=m.MyDataset(rows), collate_fn=lambda b: b, batch_size=3, num_workers=0, shuffle=True)
    ref = [[r["input_ids"] for r in b] for b in dl] + [[r["input_ids"] for r in b] for b in dl]
    assert mine == ref and len(mine) == 2 * ((len(rows) + 2) // 3)
    seq = [[r["input_ids"] for r in b] for b in m.set_dataloader(conf, m.MyDataset(rows), True)]        # for_scoring: no shuffle
    assert [x for b in seq for x in b] == [r["input_ids"] for r in rows]
