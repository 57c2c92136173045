"""Golden for the dataset preparation path (SURVEY 8(f) rank 1): the first 24 sentences of the reference's MSRA test split
(raw `sentences.txt` / `tags.txt` lines — data, ~4 KB) with the featurisation the REFERENCE produced for them, read back
from its shipped prediction pickle `data/msra/bilstm_crf_predict.pkl` (tokens, label_ids under the giga tokenizer,
max_seq_len 150), plus `data/msra/data_params.pkl` (n_sample / max_seq_len / label_size / tag2idx).  Needs /root/reference:

    python tests/golden/make_msra_sample_golden.py
"""
import json
import os
import pickle

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference/data/msra"
N = 24


if __name__ == "__main__":
    sent = open(os.path.join(REF, "test", "sentences.txt"), encoding="utf-8").read().split("\n")
    tags = open(os.path.join(REF, "test", "tags.txt"), encoding="utf-8").read().split("\n")
    pred = pickle.load(open(os.path.join(REF, "bilstm_crf_predict.pkl"), "rb"))
    dp = pickle.load(open(os.path.join(REF, "data_params.pkl"), "rb"))
    toks = [[t.decode("utf-8") for t in d["tokens"]] for d in pred]
    labs = [[int(x) for x in d["label_ids"]] for d in pred]
    vocab = sorted({c for row in toks[:N] for c in row if c not in ("[PAD]", "[UNK]")})
    out = {
        "sentences": sent[:N], "tags": tags[:N], "tokens": toks[:N], "label_ids": labs[:N],
        "giga_vocab_subset": vocab,               # enough of the giga vocabulary to tokenise the sample
        "data_params": {k: (v if not isinstance(v, dict) else {str(a): b for a, b in v.items()}) for k, v in dp.items()},
    }
    with open(os.path.join(HERE, "msra_sample.json"), "w", encoding="utf-8") as f:
        json.dump(out, f, ensure_ascii=False, indent=0)
    print(len(pred), os.path.getsize(os.path.join(HERE, "msra_sample.json")))
