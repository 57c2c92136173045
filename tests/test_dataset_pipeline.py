"""CPU: dataset preparation (.nerrec column files), the input pipeline, checkpoints and the TF tensor-bundle reader.

Golden fixtures (tests/golden/make_msra_sample_golden.py, make_variables_index_golden.py): the reference's own featurisation
of its MSRA test split, recovered from the tokens / label_ids inside `data/msra/bilstm_crf_predict.pkl`; its
`data_params.pkl`; the `variables.index` tables of its four serving checkpoints."""
import json
import os
import pickle

import numpy as np
import pytest
import torch

from chinesener_b200 import checkpoint, tf_checkpoint, variables
from chinesener_b200.data import base_preprocess as bp, preprocess, records
from chinesener_b200.data.tokenizer import TokenizerAdapter, TokenizerGiga

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SAMPLE = json.load(open(os.path.join(GOLD, "msra_sample.json"), encoding="utf-8"))


def _sample_dir(tmp_path):
    for split, n0, n1 in (("train", 0, 16), ("val", 16, 20), ("test", 0, 24)):
        d = tmp_path / "raw" / split
        d.mkdir(parents=True)
        (d / "sentences.txt").write_text("\n".join(SAMPLE["sentences"][n0:n1]) + "\n", encoding="utf-8")
        (d / "tags.txt").write_text("\n".join(SAMPLE["tags"][n0:n1]) + "\n", encoding="utf-8")
    return str(tmp_path / "raw")


def _prepare(tmp_path, vocab=None):
    tok = TokenizerAdapter(SAMPLE["giga_vocab_subset"] if vocab is None else vocab)
    proc = bp.get_instance(TokenizerGiga, preprocess.MSRA_MAX_SEQ_LEN, preprocess.MSRA_TAG2IDX, tok)
    src, out = _sample_dir(tmp_path), str(tmp_path / "out")
    emb = np.random.default_rng(0).normal(size=(len(tok.vocab2idx), 50)).astype(np.float32)
    for split in preprocess.MAPPING:
        preprocess.dump_records(proc, src, out, split, embedding=emb, verbose=False)
    return out, tok


def test_featurisation_equals_the_references_own_records(tmp_path):
    """tokens and label_ids of the sample == what the reference's pipeline wrote for the same sentences (its pickle)."""
    out, tok = _prepare(tmp_path)
    rec = records.RecordFile(os.path.join(out, "giga_predict.nerrec"))
    b = rec.batch(slice(0, rec.n))
    assert rec.n == 24 and rec.max_seq_len == 150
    assert b["tokens"] == SAMPLE["tokens"]
    assert b["label_ids"].tolist() == SAMPLE["label_ids"]
    assert b["token_ids"].dtype == torch.int32 and b["label_ids"].dtype == torch.int32       # dataset.py:23-27 casts
    # mask / seq_len / segment_ids follow format_sequence (base_preprocess.py:164-191)
    n_tok = [sum(1 for t in row if t != "[PAD]") for row in SAMPLE["tokens"]]
    assert b["seq_len"].tolist() == n_tok
    assert (b["mask"].sum(1) == b["seq_len"]).all() and int(b["segment_ids"].sum()) == 0
    pad_id = tok.vocab2idx["[PAD]"]
    assert all((b["token_ids"][i, n:] == pad_id).all() for i, n in enumerate(n_tok))
    assert b["labels"][0][:5] == [{v: k for k, v in preprocess.MSRA_TAG2IDX.items()}[i] for i in SAMPLE["label_ids"][0][:5]]


def test_out_of_vocabulary_characters_become_unk_in_the_references_records(tmp_path):
    """The sample with every tenth vocabulary character removed: exactly the positions where the reference's record holds
    a removed character become [UNK] (with the [UNK] id), everything else and every label_id stays the reference's."""
    dropped = set(SAMPLE["giga_vocab_subset"][::10])
    out, tok = _prepare(tmp_path, [c for c in SAMPLE["giga_vocab_subset"] if c not in dropped])
    b = records.RecordFile(os.path.join(out, "giga_predict.nerrec")).batch(slice(0, 24))
    want = [["[UNK]" if t in dropped else t for t in row] for row in SAMPLE["tokens"]]
    assert b["tokens"] == want and sum(row.count("[UNK]") for row in want) > 24
    assert b["label_ids"].tolist() == SAMPLE["label_ids"]
    unk = b["token_ids"] == tok.vocab2idx["[UNK]"]
    assert unk.tolist() == [[t == "[UNK]" for t in row] for row in want]


def test_data_params_match_the_shipped_pickle(tmp_path):
    out, _ = _prepare(tmp_path)
    dp = pickle.load(open(os.path.join(out, "giga_data_params.pkl"), "rb"))
    ref = SAMPLE["data_params"]
    assert dp["max_seq_len"] == ref["max_seq_len"] == 150 and dp["label_size"] == ref["label_size"] == 10
    assert dp["tag2idx"] == ref["tag2idx"] and {str(k): v for k, v in dp["idx2tag"].items()} == ref["idx2tag"]
    assert dp["n_sample"] == 16 and dp["embedding"].shape[1] == 50
    ds = records.NerDataset(out, batch_size=5, epoch_size=3, model_name="bilstm_crf")
    assert ds.params["step_per_epoch"] == 3 and ds.params["num_train_steps"] == 9              # dataset.py:62-63


def test_record_file_round_trip_with_optional_features(tmp_path):
    L, rng = 6, np.random.default_rng(1)
    feats = []
    for i in range(7):
        n = 1 + i % L
        feats.append({"tokens": ["字%d" % j for j in range(n)] + ["[PAD]"] * (L - n), "token_ids": rng.integers(0, 70000, L).tolist(),
                      "segment_ids": [0] * L, "mask": [1] * n + [0] * (L - n), "seq_len": n, "labels": ["O"] * n + ["[PAD]"] * (L - n),
                      "label_ids": [1] * n + [0] * (L - n), "label_len": n,
                      "softlexicon_ids": rng.integers(0, 704370, L * 40).tolist(), "softlexicon_weights": rng.random(L * 40).tolist()})
    path = str(tmp_path / "x.nerrec")
    records.write_records(path, feats, L)
    rec = records.RecordFile(path)
    rows = np.array([5, 0, 3])
    b = rec.batch(rows)
    assert b["tokens"] == [feats[r]["tokens"] for r in rows] and b["labels"] == [feats[r]["labels"] for r in rows]
    assert b["token_ids"].tolist() == [feats[r]["token_ids"] for r in rows]                  # > int16: stored as int32
    assert b["softlexicon_ids"].shape == (3, L * 40) and b["softlexicon_ids"].dtype == torch.int32
    np.testing.assert_allclose(b["softlexicon_weights"].numpy(), np.asarray([feats[r]["softlexicon_weights"] for r in rows], np.float32))
    assert "label_len" not in b
    with pytest.raises(ValueError):
        (tmp_path / "bad").write_bytes(b"not a record file")
        records.RecordFile(str(tmp_path / "bad"))


def test_shuffle_window_is_tf_datas_buffered_shuffle():
    rng = np.random.default_rng(0)
    order = records.shuffle_window(1000, 64, rng)
    assert sorted(order.tolist()) == list(range(1000))               # a permutation
    # element e enters the buffer when input e-63 has been consumed, so it cannot come out before output position e-63
    assert all(pos >= e - 63 for pos, e in enumerate(order))
    assert (order != np.arange(1000)).any()
    assert records.shuffle_window(10, 64, rng).tolist() != list(range(10)) or True
    assert sorted(records.shuffle_window(10, 64, rng).tolist()) == list(range(10))


def test_input_fn_batching(tmp_path):
    out, _ = _prepare(tmp_path)
    ds = records.NerDataset(out, batch_size=5, epoch_size=3, model_name="bilstm_crf")
    train = list(ds.build_input_fn("train")())
    sizes = [b["token_ids"].shape[0] for b in train]
    assert sum(sizes) == 16 * 3 and sizes[:-1] == [5] * (len(sizes) - 1) and sizes[-1] == 3   # repeat(3).batch(5): runs across epochs
    assert "tokens" not in train[0]                                   # TRAIN keeps the string features off the hot loop
    pred = list(ds.build_input_fn("predict", is_predict=True)())
    assert [b["token_ids"].shape[0] for b in pred] == [5, 5, 5, 5, 4]
    assert [t for b in pred for t in b["tokens"]] == SAMPLE["tokens"]  # ordered, one pass


def test_extract_prefix_surfix_and_optional_batch_keys():
    assert bp.extract_prefix_surfix("bert_bilstm_crf") == (None, "bert")
    assert bp.extract_prefix_surfix("bilstm_crf_softlexicon") == ("softlexicon", "giga")
    assert bp.extract_prefix_surfix("bert_bilstm_crf_softlexicon") == ("softlexicon", "bert")
    assert bp.extract_prefix_surfix("transformer_tener_crf_bichar") == ("bichar", "giga")
    assert bp.extract_prefix_surfix("bilstm_crf_ex_softword") == ("ex_softword", "giga")
    f = {"tokens": ["a"] * 3, "token_ids": [1, 2, 3], "mask": [1, 1, 0], "segment_ids": [0] * 3, "seq_len": 2, "task_ids": 1,
         "softlexicon_ids": list(range(120)), "softlexicon_weights": [0.5] * 120}
    b = bp.features_to_batch([f, dict(f, task_ids=0)])
    assert b["task_ids"].tolist() == [1, 0] and b["task_ids"].dtype == torch.int32
    assert b["softlexicon_ids"].shape == (2, 120) and b["softlexicon_weights"].dtype == torch.float32


# ----------------------------------------------------------------------------- checkpoints
def test_npz_checkpoint_keeps_adam_slots_and_global_step(tmp_path):
    from chinesener_b200.tools import train_utils
    st = variables.VariableStore("cpu", seed=3)
    st.get_variable("logits/kernel", (4, 3), variables.glorot_uniform)
    st.get_variable("logits/bias", (3,), variables.zeros)
    st.get_variable("embedding/table", (5, 2), variables.ones, trainable=False)
    fs = train_utils._flat(st)
    fs.m.copy_(torch.arange(fs.m.numel(), dtype=torch.float32))
    fs.v.copy_(torch.arange(fs.v.numel(), dtype=torch.float32) * 2)
    st.global_step = 1234
    want_m = {n: m.clone() for n, (m, v) in fs.slot_dict().items()}
    p1 = checkpoint.save_checkpoint(st, str(tmp_path), keep_checkpoint_max=2)
    for step in (1300, 1400):
        st.global_step = step
        checkpoint.save_checkpoint(st, str(tmp_path), keep_checkpoint_max=2)
    assert not os.path.exists(p1) and checkpoint.latest_checkpoint(str(tmp_path)).endswith("model.ckpt-1400.npz")
    st.global_step = 1234
    p1 = checkpoint.save_checkpoint(st, str(tmp_path), keep_checkpoint_max=5)

    st2 = variables.VariableStore("cpu", seed=9)                        # a fresh process: variables first, slots pending
    st2.get_variable("logits/kernel", (4, 3), variables.glorot_uniform)
    st2.get_variable("logits/bias", (3,), variables.zeros)
    st2.get_variable("embedding/table", (5, 2), variables.zeros, trainable=False)
    assert checkpoint.restore_checkpoint(st2, p1) == 1234 and st2.global_step == 1234
    assert torch.equal(st2.vars["logits/kernel"], st.vars["logits/kernel"]) and torch.equal(st2.vars["embedding/table"], torch.ones(5, 2))
    fs2 = train_utils._flat(st2)                                          # the train op builds the flat state: slots land
    for n, (m, v) in fs2.slot_dict().items():
        assert torch.equal(m, want_m[n]) and torch.equal(v, want_m[n] * 2)
    # a changed trainable set rebuilds the flat state; moments of surviving variables carry over (by name)
    st2.get_variable("crf_layer/transitions", (3, 3), variables.xavier)
    fs3 = train_utils._flat(st2)
    assert fs3 is not fs2 and torch.equal(fs3.slot_dict()["logits/bias"][0], want_m["logits/bias"])
    assert float(fs3.slot_dict()["crf_layer/transitions"][0].abs().sum()) == 0.0


def test_tf_bundle_index_reader_on_the_references_serving_checkpoints(tmp_path):
    gold = json.load(open(os.path.join(GOLD, "variables_index.json")))
    for model, g in gold.items():
        header, entries = tf_checkpoint.read_bundle_index(os.path.join(GOLD, "variables_index", model + ".index"), verify=True)
        assert header["num_shards"] == 1
        assert {k: {"dtype": e["dtype"], "shape": e["shape"]} for k, e in entries.items()} == g["variables"]
        assert sum(e["size"] for e in entries.values()) == g["total_bytes"]
        assert list(entries) == sorted(entries, key=lambda s: s.encode())            # table order
    _, e = tf_checkpoint.read_bundle_index(os.path.join(GOLD, "variables_index", "bert_bilstm_crf.index"))
    assert len(e) == 207 and sum(v["size"] for v in e.values()) == 412755392                 # BASELINE.md §1
    assert e["bilstm_layer/bidirectional_rnn/fw/multi_rnn_cell/cell_0/lstm_cell/kernel"]["shape"] == [896, 512]
    assert e["global_step"]["dtype"] == tf_checkpoint.DT_INT64 and e["global_step"]["shape"] == []
    import shutil
    prefix = str(tmp_path / "lfs")                                                     # the data file is an LFS pointer upstream
    open(prefix + ".data-00000-of-00001", "wb").write(b"version https://git-lfs.github.com/spec/v1\n")
    shutil.copyfile(os.path.join(GOLD, "variables_index", "bilstm_crf.index"), prefix + ".index")
    with pytest.raises(ValueError):
        tf_checkpoint.load_tf_checkpoint(prefix)


def test_tf_bundle_write_read_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    tensors = {"bert/embeddings/word_embeddings": rng.normal(size=(50, 8)).astype(np.float32), "global_step": np.asarray(77, np.int64),
               "crf_layer/transitions": rng.normal(size=(10, 10)).astype(np.float32)}
    for i in range(200):                                               # several data blocks + prefix-compressed keys
        tensors[f"bert/encoder/layer_{i}/attention/self/query/kernel"] = rng.normal(size=(3, 3)).astype(np.float32)
    prefix = str(tmp_path / "bert_model.ckpt")
    tf_checkpoint.save_tf_checkpoint(prefix, tensors)
    out = tf_checkpoint.load_tf_checkpoint(prefix, verify=True)
    assert set(out) == set(tensors) and all(np.array_equal(out[k], tensors[k]) and out[k].dtype == tensors[k].dtype for k in tensors)
    assert tf_checkpoint.crc32c(b"123456789") == 0xE3069283                             # the CRC-32C check value
    assert tf_checkpoint.find_checkpoint(str(tmp_path)) == prefix and tf_checkpoint.find_checkpoint(str(tmp_path / "nope")) is None


def test_load_bert_checkpoint_assigns_by_name_and_fails_loudly(tmp_path):
    from chinesener_b200 import bert
    cfg = {'vocab_size': 30, 'hidden_size': 8, 'num_hidden_layers': 1, 'num_attention_heads': 2, 'intermediate_size': 16,
           'max_position_embeddings': 12, 'type_vocab_size': 2}
    with pytest.raises(FileNotFoundError):                     # a pretrain_dir without bert_config.json: the reference fails too
        bert.load_bert_config(str(tmp_path / "missing"))
    d = tmp_path / "ch"
    d.mkdir()
    (d / "bert_config.json").write_text(json.dumps(cfg))
    src = variables.VariableStore("cpu", seed=11)
    bert.create_bert_variables(dict(bert.BERT_BASE_CHINESE, **cfg), src)
    tf_checkpoint.save_tf_checkpoint(str(d / "bert_model.ckpt"), {k: v.numpy() for k, v in src.state_dict().items()})
    dst = variables.VariableStore("cpu", seed=99)
    bert.create_bert_variables(bert.load_bert_config(str(d)), dst)         # creation triggers load_bert_checkpoint(pretrain_dir)
    assert all(torch.equal(dst.vars[k], src.vars[k]) for k in src.vars)
    d2 = tmp_path / "random"
    d2.mkdir()
    (d2 / "bert_config.json").write_text(json.dumps(cfg))
    with pytest.warns(UserWarning, match="random"):
        bert.create_bert_variables(bert.load_bert_config(str(d2)), variables.VariableStore("cpu", seed=1))


def _msr_dir(tmp_path, rng):
    """the sample sentences re-cut into random words, in the msr_<split>.utf8 layout (words separated by two spaces)."""
    d = tmp_path / "msr_raw"
    d.mkdir()
    for split, n0, n1 in (("training", 0, 10), ("test_gold", 10, 13), ("test", 13, 18)):
        lines = []
        for s in SAMPLE["sentences"][n0:n1]:
            chars, words, i = s.split(" "), [], 0
            while i < len(chars):
                k = int(rng.integers(1, 4))
                words.append("".join(chars[i:i + k]))
                i += k
            lines.append("  ".join(words))
        (d / "msr_{}.utf8".format(split)).write_text("\n".join(lines) + "\n\n", encoding="utf-8")
    return str(d)


def test_msr_word_segmentation_tags(tmp_path):
    """data/msr/preprocess.py:27-52: a word of n characters -> S | B E | B I.. E; the sentence is its characters."""
    assert [preprocess.msr_gen_tag(n) for n in (1, 2, 3, 5)] == ["S", "B E", "B I E", "B I I I E"]
    (tmp_path / "msr_test.utf8").write_text("“  人们  常  说  生活是  一\n\n", encoding="utf-8")
    s, t = preprocess.load_msr_data(str(tmp_path), "test")
    assert s == ["“ 人 们 常 说 生 活 是 一"] and t == ["S B E S S B I E S"]


def _prepare_two_tasks(tmp_path, tokenizer_type=TokenizerGiga, L=preprocess.MSRA_MAX_SEQ_LEN):
    vocab = list(SAMPLE["giga_vocab_subset"]) + (["[CLS]", "[SEP]"] if tokenizer_type != TokenizerGiga else [])
    tok = TokenizerAdapter(vocab)
    root = tmp_path / "data"
    src = _sample_dir(tmp_path)
    ner = bp.get_instance(tokenizer_type, L, preprocess.MSRA_TAG2IDX, tok)
    for split in preprocess.MAPPING:
        preprocess.dump_records(ner, src, str(root / "msra"), split, verbose=False)
    cws = bp.get_instance(tokenizer_type, L, preprocess.MSR_TAG2IDX, tok)
    msr_src = _msr_dir(tmp_path, np.random.default_rng(3))
    for split in preprocess.MSR_MAPPING:
        preprocess.dump_records(cws, msr_src, str(root / "msr"), split, mapping=preprocess.MSR_MAPPING, verbose=False,
                                load_data=preprocess.load_msr_data)
    return str(root), tok


def test_multi_dataset_interleaves_sample_by_sample(tmp_path):
    """dataset.py:73-141: choose_from_datasets(range(2).repeat()) -> tasks alternate 0,1,0,1 until the shorter dataset runs
    out, then the longer one alone; repeat(epoch).batch(B); params carry each dataset's own params + task_list."""
    root, _ = _prepare_two_tasks(tmp_path)
    md = records.MultiDataset(root, ["msra", "msr"], batch_size=4, epoch_size=2, model_name="bilstm_crf_mtl")
    p = md.params
    assert p["task_list"] == ["msra", "msr"] and p["max_seq_len"] == 150
    assert p["msra"]["label_size"] == 10 and p["msr"]["label_size"] == 7 and p["msr"]["idx2tag"][4] == "S"
    assert p["step_per_epoch"] == 16 // 4 and p["num_train_steps"] == 2 * 4          # max over the datasets (16 vs 10 samples)
    train = list(md.build_input_fn("train")())
    tasks = np.concatenate([b["task_ids"].numpy() for b in train])
    assert train[0]["task_ids"].dtype == torch.int32 and tasks.shape == (2 * 26,)
    per_epoch = [0, 1] * 10 + [0] * 6                                             # 10 msr + 16 msra sentences
    assert tasks.tolist() == per_epoch * 2
    sizes = [b["token_ids"].shape[0] for b in train]
    assert sizes == [4] * 13                                                        # 52 = 13 * 4: batches run across the epoch boundary
    # every sentence of both datasets appears once per epoch (shuffle is a permutation), labels stay inside the task's tag set
    lab = torch.cat([b["label_ids"] for b in train])
    assert int(lab[torch.from_numpy(tasks == 1)].max()) <= 6
    epoch0 = torch.cat([b["token_ids"] for b in train])[:26]
    seen = sorted(tuple(r.tolist()) for r in epoch0[torch.from_numpy(tasks[:26] == 1)])
    rec = records.RecordFile(os.path.join(root, "msr", "giga_train.nerrec"))
    assert seen == sorted(tuple(r.tolist()) for r in rec.batch(slice(0, rec.n), with_strings=False)["token_ids"])
    # EVAL pass: ordered, one pass
    ev = list(md.build_input_fn("valid", is_predict=True)())
    assert np.concatenate([b["task_ids"].numpy() for b in ev]).tolist() == [0, 1, 0, 1, 0, 1, 0]
    # per-dataset PREDICT pass keeps the dataset's order and its task id
    pr = list(md.build_predict_fn("msr")())
    assert sum(b["token_ids"].shape[0] for b in pr) == 5 and all((b["task_ids"] == 1).all() for b in pr)
    assert "tokens" in pr[0] and pr[0]["tokens"][0][0] == SAMPLE["sentences"][13].split(" ")[0]
