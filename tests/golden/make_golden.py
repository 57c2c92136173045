"""Generate the golden fixtures under tests/golden/ from the reference's shipped artefacts.

Run in the authoring container (needs /root/reference, read-only):  python tests/golden/make_golden.py
Outputs (committed):
  predict_pickle_stats.json   per shipped *_predict.pkl: #sentences, #non-zero pred_ids on [PAD]
                              tokens (pins crf_decode's zero-fill), entity micro / weighted F1 by
                              chinesener_b200.evaluation (pins the evaluator against BASELINE.md §2)
  msra_bert_bilstm_crf_sample.pkl   first 48 sentences of data/msra/bert_bilstm_crf_predict.pkl

`python tests/golden/make_golden.py --sample-reports` needs only the committed sample and scikit-learn:
  msra_bert_bilstm_crf_sample_reports.json   the sample's tag-level report by scikit-learn (the library the reference's
                              evaluation.py:38-46 uses for it) and its entity-level counts and F1
"""
import glob
import json
import os
import pickle
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = "/root/reference"

from chinesener_b200 import evaluation  # noqa: E402


def main():
    stats = {}
    for data in ("msra", "people_daily"):
        idx2tag = pickle.load(open(f"{REF}/data/{data}/data_params.pkl", "rb"))["idx2tag"]
        for path in sorted(glob.glob(f"{REF}/data/{data}/*_predict.pkl")):
            name = os.path.basename(path)[:-len("_predict.pkl")]
            if name == "MRC":
                continue
            pred = pickle.load(open(path, "rb"))
            viol = 0
            for s in pred:
                for tok, p in zip(s["tokens"], s["pred_ids"]):
                    if tok == b"[PAD]" and p != 0:
                        viol += 1
            ent = evaluation.SingleEval(pred, idx2tag).entity_eval()
            stats[f"{data}/{name}"] = {
                "n": len(pred), "pad_violations": viol,
                "micro_f1": round(ent["micro avg"]["f1-score"], 4), "weighted_f1": round(ent["weighted avg"]["f1-score"], 4),
                "support": ent["micro avg"]["support"]}
            print(name, stats[f"{data}/{name}"], flush=True)
    out = os.path.join(ROOT, "tests", "golden")
    json.dump({"idx2tag_msra": {int(k): v for k, v in pickle.load(open(f"{REF}/data/msra/data_params.pkl", "rb"))["idx2tag"].items()},
               "stats": stats}, open(os.path.join(out, "predict_pickle_stats.json"), "w"), indent=1, ensure_ascii=False)
    pred = pickle.load(open(f"{REF}/data/msra/bert_bilstm_crf_predict.pkl", "rb"))[:48]
    sample = [{"pred_ids": [int(x) for x in s["pred_ids"]], "label_ids": [int(x) for x in s["label_ids"]],
               "tokens": [t.decode() for t in s["tokens"]]} for s in pred]
    pickle.dump(sample, open(os.path.join(out, "msra_bert_bilstm_crf_sample.pkl"), "wb"))


def sample_reports():
    from sklearn.metrics import precision_recall_fscore_support
    from chinesener_b200.tools.predict_utils import process_prediction
    out = os.path.join(ROOT, "tests", "golden")
    idx2tag = {int(k): v for k, v in json.load(open(os.path.join(out, "predict_pickle_stats.json")))["idx2tag_msra"].items()}
    sample = [process_prediction(dict(s), idx2tag) for s in pickle.load(open(os.path.join(out, "msra_bert_bilstm_crf_sample.pkl"), "rb"))]
    y_true = [int(t) for s in sample for t in s["label_ids"]]
    y_pred = [int(t) for s in sample for t in s["pred_ids"]]
    labels = [k for k, v in sorted(idx2tag.items()) if v not in ("[PAD]", "[CLS]", "[SEP]")]
    p, r, f, n = precision_recall_fscore_support(y_true, y_pred, labels=labels, average=None, zero_division=0)
    wp, wr, wf, _ = precision_recall_fscore_support(y_true, y_pred, labels=labels, average="weighted", zero_division=0)
    tag = {str(lab): {"precision": float(p[i]), "recall": float(r[i]), "f1-score": float(f[i]), "support": int(n[i])}
           for i, lab in enumerate(labels)}
    tag["weighted avg"] = {"precision": float(wp), "recall": float(wr), "f1-score": float(wf)}
    ent = evaluation.entity_report([s["labels"] for s in sample], [s["preds"] for s in sample])
    json.dump({"n_tokens": len(y_true), "tag_report_sklearn": tag, "entity_report": ent},
              open(os.path.join(out, "msra_bert_bilstm_crf_sample_reports.json"), "w"), indent=1)


if __name__ == "__main__":
    if "--sample-reports" in sys.argv:
        sample_reports()
    else:
        main()
