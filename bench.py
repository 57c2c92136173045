"""bench.py — sentences/sec of the bert_bilstm_crf hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (sm_100a kernels)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path (oracle port)
  ... --dump-outputs DIR                                    also write the pred_ids of the last timed step(s) to DIR/*.npy

One "step" = one PREDICT pass of model.bert_bilstm_crf.build_graph over one synthetic
MSRA-shaped batch (BERT-base encoder -> BiLSTM -> logits -> CRF log-likelihood + Viterbi),
B=64 sentences per GPU, L=128 — BASELINE.json configs[2].  N>1: one process per GPU under
torchrun, batches sharded across ranks, no data-path collective (decode shards by sentence);
timing = CUDA events, max over ranks.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, SEQ_LEN, LABELS = 64, 128, 10
METRIC = "sentences/sec bert_bilstm_crf MSRA L=128"
WORKLOAD = ("bert_bilstm_crf msra seq_len=128 bs=64/GPU PREDICT step: BERT-base fwd (12L, H768) + BiLSTM(H128, relu) "
            "+ logits + CRF Viterbi -> pred_ids (the log-likelihood is part of the graph but PREDICT does not fetch it, as "
            "in the reference's Estimator); bf16 tcgen05 GEMM operands, fp32 residual/LSTM/CRF; MSRA-shaped lengths")


def dump_outputs(dirname, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, as float32 (the tags are small integers, exact in float32), so that
    two builds run with the same arguments can be compared output for output."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a, dtype=np.float32))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1400.0, "fallback"


class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed regions (B200_PROFILING.md recipe).  NVML is polled
    from a thread every ~2 ms (the timed regions last tens of ms, shorter than one `nvidia-smi -lms` period);
    `nvidia-smi` is the fallback when the NVML binding is unavailable."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.h, self.stop_flag = index, [], None, None, False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)

    def start(self):
        try:
            self.nv, self.h = self._nvml_handle()
            self.mx = float(self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.h = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")]
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.rows.append((sm, [n for b, n in bits if r & b], util))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.h is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            # host-only stretches between the GPU-timed regions (building tables / estimators) would dilute the median
            # with idle-clock samples: take it over the samples NVML reports as busy (utilisation window >= 10 %)
            busy = [r for r in self.rows if r[2] >= 10]
            rows = busy if len(busy) >= 20 else self.rows
            sm = [r[0] for r in rows]
            reasons = sorted({n for r in self.rows for n in r[1]})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.rows), "samples_under_load": len(busy), "source": "nvml, 2 ms poll from the first device-resident timed step to the last kernel-roofline launch"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi -lms 20"}


def bind_to_gpu_numa_node(index):
    """One process per GPU: run this rank's host threads on the CPUs NVML reports as local to its GPU
    (kernel launches and pinned-memory copies from the far socket are what made single ranks straggle at N=8)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return {"cpus_before": before, "cpus_after": len(os.sched_getaffinity(0))}
    except Exception as e:      # no NVML / restricted cpuset: keep the inherited affinity
        return {"error": str(e)[:80]}


def make_estimator():
    from chinesener_b200 import engine, synthetic
    params = dict(synthetic.data_params(SEQ_LEN, LABELS), pretrain_dir="")
    est = engine.Estimator("bert_bilstm_crf", params)
    return est


def host_batches(n, seed0):
    from chinesener_b200 import synthetic
    out = []
    for i in range(n):
        f = synthetic.msra_batch(B_PER_GPU, SEQ_LEN, seed=seed0 + i)
        out.append({k: v.pin_memory() for k, v in f.items()})
    return out


def oracle_weights_and_params(seed=1234):
    """Random-init TF-named weights on the CPU for the reference arm / cpu_baseline."""
    from chinesener_b200 import synthetic, variables
    from chinesener_b200.bert import create_bert_variables
    from chinesener_b200.config import BERT_BASE_CHINESE
    st = variables.VariableStore("cpu", seed=seed)
    create_bert_variables(BERT_BASE_CHINESE, st)
    D, H = 768, 128
    for d in ("fw", "bw"):
        st.get_variable(f"bilstm_layer/bidirectional_rnn/{d}/multi_rnn_cell/cell_0/lstm_cell/kernel", (D + H, 4 * H), variables.glorot_uniform)
        st.get_variable(f"bilstm_layer/bidirectional_rnn/{d}/multi_rnn_cell/cell_0/lstm_cell/bias", (4 * H,), variables.zeros)
    st.get_variable("logits/kernel", (2 * H, LABELS), variables.glorot_uniform)
    st.get_variable("logits/bias", (LABELS,), variables.zeros)
    st.get_variable("crf_layer/transitions", (LABELS, LABELS), variables.xavier)
    params = dict(synthetic.data_params(SEQ_LEN, LABELS), rnn_activation="relu")
    return st.state_dict(), params


_CPU_THREADS = None


def pick_cpu_threads():
    """Thread count that maximises the reference's CPU throughput on this host.

    TF's default on CPU is "all cores" (tools/utils.py:33-40 caps threads only under --gpu); on a
    many-core host the small per-op matrices of an L=128 batch run slower oversubscribed, so a
    1-second fp32 GEMM probe (the dominant op: [n_tok,768]x[768,3072]) picks the best of
    {all, 64, 32, 16} and the choice is reported as `cores`.
    """
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, 64, 32, 16) if c <= ncpu}, reverse=True)
    a, b = torch.randn(2048, 768), torch.randn(768, 3072)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.perf_counter()
        for _ in range(5):
            a @ b
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    _CPU_THREADS = best
    return best


def time_cpu_reference(weights, params, host_batches_, reps=2):
    """The reference's CPU path (PyTorch-CPU fp32 restatement; TF 1.14 is not installable) on the host cores, over the
    SAME 64-sentence host batches and the SAME weights the GPU arm was timed on.  -> (sentences/s, rep seconds, outputs of
    the first timed batch): the outputs are the checker of `parity_checked`."""
    from oracle import models as omodels
    torch.set_num_threads(pick_cpu_threads())
    small = {k: (v[:8] if torch.is_tensor(v) else v) for k, v in host_batches_[0].items()}
    with torch.no_grad():
        omodels.bert_bilstm_crf(weights, small, params, dtype=torch.float32)        # warms the thread pool / allocator
    ts, first = [], None
    for r in range(reps):
        feats = host_batches_[r % len(host_batches_)]
        t0 = time.perf_counter()
        with torch.no_grad():
            out = omodels.bert_bilstm_crf(weights, feats, params, dtype=torch.float32)
        ts.append(time.perf_counter() - t0)
        if first is None:
            first = out
    n_sent = host_batches_[0]['token_ids'].shape[0]
    return n_sent / float(np.median(ts)), ts, first


def check_parity(est, feats, oracle_out):
    """pred_ids of one TIMED batch against the oracle, outside every timed region.
    (1) Viterbi tags from Estimator.predict must equal, bit for bit, the oracle's Viterbi run on the CUDA path's own fp32
        emission logits (integer output);  (2) tag agreement with the end-to-end fp32 CPU oracle (its own logits) and the
        max |logit| distance to it are reported as numbers (bf16 operands vs fp32: not expected to be bit-equal)."""
    from chinesener_b200 import variables
    from chinesener_b200.tools import layer
    from oracle import crf as ocrf
    dev = est.to_device(feats)
    pred = est.predict(feats)['pred_ids'].numpy()
    with variables.use_store(est.store):
        emb = layer.pretrain_bert_embedding(dev['token_ids'], dev['mask'], dev['segment_ids'], est.params['pretrain_dir'], 0.1, False)
        x = layer.bilstm(emb, 'lstm', est.params['rnn_activation'], est.params['hidden_units_list'], [1.0], 1, dev['seq_len'], 'float32', False)
        logits = layer.dense(x, LABELS, 'logits')
    torch.cuda.synchronize()
    lg = logits.cpu().numpy()
    trans = est.store.vars['crf_layer/transitions'].cpu().numpy()
    lens = feats['seq_len'].numpy()
    ref_pred, _ = ocrf.crf_decode(lg, trans, lens, dtype=np.float32)
    valid = np.arange(SEQ_LEN)[None, :] < lens[:, None]
    bit_exact = bool(np.array_equal(pred, ref_pred))
    agree = float((pred == oracle_out['pred_ids'])[valid].mean())
    err = float(np.abs(lg - oracle_out['logits'].numpy())[valid].max())
    scale = float(np.abs(oracle_out['logits'].numpy())[valid].max())
    # the bar: integer output bit-exact; bf16-operand emission logits within 2e-2 of the logit scale of the fp32 CPU oracle
    # (tests/test_timed_config_gpu.py holds the tighter 1e-2 bar against the oracle evaluated with the same bf16 rounding
    # points); the tag agreement with the end-to-end fp32 oracle is reported as a number — near-tie paths flip under bf16
    return {"parity_checked": bool(bit_exact and err <= 2e-2 * max(1.0, scale)), "viterbi_bit_exact_on_cuda_logits": bit_exact,
            "tag_agreement_with_cpu_oracle": agree, "max_abs_logit_diff_vs_fp32_cpu_oracle": err,
            "max_abs_logit": float(np.abs(oracle_out['logits'].numpy())[valid].max()),
            "what": "batch 0 of the timed batches; Estimator.predict tags == oracle Viterbi on the CUDA logits (bit-exact), "
                    "and vs the PyTorch-CPU fp32 oracle end to end (rate); checked outside the timed regions"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_sent = B_PER_GPU           # the same 64-sentence batch our arm steps over
    per_step = []
    from chinesener_b200 import synthetic
    from oracle import models as omodels
    torch.set_num_threads(pick_cpu_threads())
    w, params = oracle_weights_and_params()
    for i in range(args.warmup + args.steps):
        feats = synthetic.msra_batch(n_sent, SEQ_LEN, seed=1000 + i)
        t0 = time.perf_counter()
        with torch.no_grad():
            out = omodels.bert_bilstm_crf(w, feats, params, dtype=torch.float32)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            per_step.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pred_ids": np.asarray(out["pred_ids"])})
    total = float(sum(per_step))
    value = n_sent * len(per_step) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "sentences/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(per_step), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": n_sent, "seq_len": SEQ_LEN,
                   "note": "each step = one 64-sentence batch of the same workload on the host cores"},
        "cpu_baseline": {"value": value, "unit": "sentences/sec", "cores": pick_cpu_threads(), "host_cpus": os.cpu_count(), "kind": "port",
                         "sample": f"{len(per_step)} steps x {n_sent} sentences, PyTorch-CPU fp32 restatement "
                                   f"(oracle/models.py) of model/bert_bilstm_crf.py; TF 1.14 not installable"},
        "e2e": {"value": value, "unit": "sentences/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _time_launches(fn, warm=3, iters=10, flush=None, park=False):
    """Average CUDA-event duration (ms) of `fn`'s launches on the current stream: >= 3 warm-ups, a synchronize on both
    sides, optional untimed L2 flush before every timed launch.  park=True (single-kernel rooflines): the GPU waits behind
    a spin kernel while the launches are enqueued.  -> (mean_ms, min_ms)."""
    for _ in range(max(warm, 3)):
        fn()
    torch.cuda.synchronize()
    # the launches come from Python (allocation + ctypes + launch, tens of us each): park the GPU behind a spin kernel so
    # that they are all enqueued before the first one runs and every event pair brackets execution, not launch latency
    if park:
        torch.cuda._sleep(6_000_000)
    evs = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        evs.append((s, e))
    torch.cuda.synchronize()
    ts = [s.elapsed_time(e) for s, e in evs]
    return float(np.mean(ts)), float(min(ts))


def crf_sample_check(x, tr, lens, tags, ll, pred, n=2048, seed=4321):
    """Checker of the roofline-sized CRF launches (outside every timed region).  With the C restatement of the oracle
    (oracle/crf_c.c, built by __graft_entry__.build()) EVERY row the kernels processed is re-run on the host cores;
    without it, `n` rows sampled with a fixed seed go through the numpy restatement.  Viterbi tags must be bit-equal
    (integer output); the log-likelihood must agree with the fp64 oracle within 1e-4 relative + 1e-4 absolute (the
    tolerance of tests/test_crf_gpu.py).  Takes tensors on any device."""
    from oracle import crf as ocrf, native as onative
    B = x.shape[0]
    t = tr.cpu().numpy()
    if onative.available():
        xs, ls, ys = x.cpu().numpy(), lens.cpu().numpy(), tags.cpu().numpy()
        t0 = time.perf_counter()
        ref_pred, _ = onative.crf_decode(xs, t, ls)
        t1 = time.perf_counter()
        ref_ll = onative.crf_log_likelihood(xs, ys, ls, t)
        t2 = time.perf_counter()
        got_pred, got_ll = pred.cpu().numpy(), ll.cpu().numpy()
        how = {"checker": "oracle/crf_c.c (plain C, OpenMP) on every row", "cpu_decode_s": t1 - t0, "cpu_loglik_s": t2 - t1,
               "cpu_threads": os.cpu_count()}
    else:
        idx = torch.from_numpy(np.sort(np.random.RandomState(seed).choice(B, size=min(n, B), replace=False))).to(x.device)
        xs, ls = x.index_select(0, idx).cpu().numpy(), lens.index_select(0, idx).cpu().numpy()
        ref_pred, _ = ocrf.crf_decode(xs, t, ls, dtype=np.float32)
        ref_ll = ocrf.crf_log_likelihood(xs, tags.index_select(0, idx).cpu().numpy(), ls, t)
        got_pred, got_ll = pred.index_select(0, idx).cpu().numpy(), ll.index_select(0, idx).cpu().numpy()
        how = {"checker": "oracle/crf.py (numpy) on rows sampled with a fixed seed"}
    return dict(how, rows_checked=int(ref_pred.shape[0]), rows_launched=int(B),
                viterbi_bit_exact=bool(np.array_equal(got_pred, ref_pred)),
                viterbi_rows_differing=int((got_pred != ref_pred).any(axis=1).sum()),
                loglik_max_rel_err_vs_fp64=float(np.max(np.abs(got_ll - ref_ll) / (np.abs(ref_ll) + 1.0))),
                loglik_within_tolerance=bool(np.allclose(got_ll, ref_ll, rtol=1e-4, atol=1e-4)),
                what="inputs and outputs of one untimed launch of each roofline-sized kernel vs the oracle")


def crf_rooflines(hbm_peak, peak_src, B=262144, L=128, K=LABELS):
    """SURVEY 8(d) "CRF kernel roofline run": B = 262 144 sequences, L = 128, K = 10, full lengths (1.34 GB of emission
    logits >> 126 MB L2, so every launch is L2-cold by construction).  Algorithmic bytes per sentence (SURVEY 8(d)):
    forward-alpha L*(4K+4)+8, Viterbi read L*4K+4 + write L*4+4 (backpointers stay on chip and are not counted)."""
    from chinesener_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.randn(B, L, K, device="cuda", generator=g)
    tr = torch.randn(K, K, device="cuda", generator=g) * 0.5
    lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
    tags = torch.randint(0, K, (B, L), device="cuda", dtype=torch.int32, generator=g)
    out = {}
    for key, fn, byts in (
            ("roofline_crf_fwd", lambda: ops.crf_loglik_fwd(x, tags, lens, tr), B * L * (4 * K + 4) + 8 * B + 4 * K * K),
            ("roofline_crf_viterbi", lambda: ops.crf_viterbi(x, lens, tr), B * L * 4 * K + 4 * B + 4 * K * K + B * L * 4 + 4 * B)):
        ms, best = _time_launches(fn, warm=3, iters=10, park=True)
        gbs = byts / (ms * 1e-3) / 1e9
        out[key] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": None,
                    "ms_per_launch": ms, "best_ms": best, "algorithmic_bytes_per_launch": byts, "launches_timed": 10,
                    "workload": f"B={B} L={L} K={K} full lengths, fp32 logits (working set 1.5 GB >> L2)", "peak_source": peak_src}
    try:        # untimed: the outputs of one more launch of each kernel against the oracle (every row with the C oracle)
        chk = crf_sample_check(x, tr, lens, tags, ops.crf_loglik_fwd(x, tags, lens, tr)[0], ops.crf_viterbi(x, lens, tr))
        out["roofline_crf_viterbi"]["parity_checked"] = chk["viterbi_bit_exact"]
        out["roofline_crf_fwd"]["parity_checked"] = chk["loglik_within_tolerance"]
        out["crf_roofline_parity"] = chk
    except Exception as exc:      # the checker must never cost the line its timings
        out["crf_roofline_parity"] = {"error": repr(exc)[:200]}
    del x, tags
    torch.cuda.empty_cache()
    return out


def softlexicon_roofline(hbm_peak, peak_src, flush, V=704370, E=50, L=128):
    """SoftLexicon gather-and-pool (SURVEY a12 / 8(d)): config 4's [704 370, 50] fp32 table (140.9 MB > L2), 40 slots per
    token.  `dense`: every slot a random word (the 8(d) upper bound, 9 120 B/token); `realistic`: the slot statistics of
    the reference's warm-up record (a few words per token, empty sets hold <None>, the rest <PAD> with weight 0 — rows the
    kernel never fetches).  Algorithmic bytes = 40*(4+4) ids/weights + nnz*4E gathered rows + 4*4E output, nnz counted
    from the generated weights.  L2 flushed (untimed) before every timed launch."""
    from chinesener_b200 import ops, synthetic
    g = torch.Generator(device="cuda").manual_seed(7)
    table = torch.nn.functional.normalize(torch.randn(V, E, device="cuda", generator=g), dim=1).contiguous()
    res = {}
    for B in (B_PER_GPU, 2048):
        for realistic in (False, True):
            ids, w = synthetic.softlexicon_features_device(B * L, V, realistic=realistic, seed=11)
            out = torch.empty((B * L, 4 * E), dtype=torch.float32, device="cuda")
            nnz = int((w != 0).sum())
            byts = B * L * (40 * 8 + 4 * E * 4) + nnz * E * 4
            ms, best = _time_launches(lambda: ops.softlexicon_pool(table, ids, w, 4, 10, out=out), warm=3, iters=10, flush=flush, park=True)
            gbs = byts / (ms * 1e-3) / 1e9
            res[f"{'realistic' if realistic else 'dense'}_B{B}"] = {
                "achieved": gbs, "frac": gbs / hbm_peak, "ms_per_launch": ms, "best_ms": best, "algorithmic_bytes_per_launch": byts,
                "nonzero_slots_per_token": nnz / (B * L)}
    head = res["dense_B2048"]
    return {"bound": "hbm", "achieved": head["achieved"], "peak": hbm_peak, "unit": "GB/s", "frac": head["frac"], "traffic": None,
            "headline": "dense_B2048 (262 144 tokens per launch; B=64 launches last a few us and are launch-latency bound)",
            "table": [V, E], "variants": res, "peak_source": peak_src}


def other_configs(steps, flush):
    """PREDICT sentences/s of BASELINE configs 2, 4, 5 (device-resident batches, L2 flushed between timed steps, CUDA
    events per step) — config 3 is the line's `value`."""
    from chinesener_b200 import engine, synthetic
    out = {}
    g = torch.Generator().manual_seed(5)
    char = torch.nn.functional.normalize(torch.randn(11329, 50, generator=g), dim=1).numpy()

    def run(name, est, feats, B):
        dev = est.to_device({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in feats.items()})
        fn = lambda: est.predict_device(dev)
        ms, best = _time_launches(fn, warm=3, iters=steps, flush=flush)
        out[name]["value"], out[name]["unit"], out[name]["ms_per_step"] = B / (ms * 1e-3), "sentences/sec", ms
        out[name]["best_ms"] = best

    # config 2: bert_crf msra seq_len=128 bs=32 fp32 (split-bf16 dense + fp32 attention/LayerNorm: the 1e-3 mode)
    B, L = 32, 128
    out["config2_bert_crf_fp32"] = {"workload": "bert_crf msra seq_len=128 bs=32, bert_precision='fp32' (3 bf16 tcgen05 GEMMs per dense "
                                                "layer, fp32 attention), MSRA-shaped lengths, PREDICT", "dtype": "f32 (split bf16)"}
    est = engine.Estimator("bert_crf", dict(synthetic.data_params(L, LABELS), pretrain_dir="", bert_precision="fp32"))
    run("config2_bert_crf_fp32", est, synthetic.msra_batch(B, L, seed=21), B)
    del est
    # config 4: bilstm_crf_softlexicon seq_len=128 bs=64, [704 370, 50] lexicon table
    B, L, NW = 64, 128, 704370
    out["config4_bilstm_crf_softlexicon"] = {"workload": "bilstm_crf_softlexicon seq_len=128 bs=64: B/M/E/S gather-and-pool over the "
                                                         "[704370,50] table (realistic slot statistics) + BiLSTM(200, tanh) + CRF, PREDICT",
                                             "dtype": "f32 (bf16 LSTM input projection)"}
    feats = synthetic.msra_batch(B, L, vocab=11329, seed=22)
    ids, w = synthetic.softlexicon_features_device(B * L, NW, realistic=True, seed=23)
    valid = (torch.arange(L)[None, :] < feats['seq_len'][:, None]).reshape(B * L, 1)
    feats['softlexicon_ids'] = torch.where(valid, ids.cpu(), torch.zeros_like(ids.cpu())).view(B, L * 40)
    feats['softlexicon_weights'] = (w.cpu() * valid).view(B, L * 40)
    wemb = torch.nn.functional.normalize(torch.randn(NW, 50, generator=g), dim=1).numpy()
    est = engine.Estimator("bilstm_crf_softlexicon", dict(synthetic.data_params(L, LABELS), embedding=char, word_embedding=wemb,
                                                          word_enhance_dim=4, max_lexicon_len=10))
    run("config4_bilstm_crf_softlexicon", est, feats, B)
    del est, wemb
    # config 5: transformer_tener_crf_bichar seq_len=256 bs=32
    B, L, NB = 32, 256, 300000
    out["config5_transformer_tener_crf_bichar"] = {"workload": "transformer_tener_crf_bichar msra seq_len=256 bs=32: char|bichar embedding -> "
                                                               "2 TENER layers (relative-position attention, d=160, 8 heads) + CRF, PREDICT",
                                                   "dtype": "f32 (split bf16 dense)"}
    feats = synthetic.msra_batch(B, L, vocab=11329, seed=24)
    feats['bichar_ids'] = torch.randint(0, NB, (B, L), generator=g, dtype=torch.int32)
    bemb = torch.nn.functional.normalize(torch.randn(NB, 50, generator=g), dim=1).numpy()
    est = engine.Estimator("transformer_tener_crf_bichar", dict(synthetic.data_params(L, LABELS), embedding=char, bichar_embedding=bemb))
    run("config5_transformer_tener_crf_bichar", est, feats, B)
    del est
    torch.cuda.empty_cache()
    return out


class GemmTimer:
    """Per-launch CUDA-event timing of the dominant kernel (tcgen05 GEMM) on the launching stream."""

    def __init__(self):
        self.recs = []

    @contextlib.contextmanager
    def __call__(self, name, flops):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        yield
        e.record()
        self.recs.append((s, e, flops))

    def summary(self):
        torch.cuda.synchronize()
        ms = sum(s.elapsed_time(e) for s, e, _ in self.recs)
        fl = sum(f for _, _, f in self.recs)
        return ms, fl, len(self.recs)


def run_ours(args):
    from chinesener_b200 import _lib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sm_100a kernels have no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None   # N=1 keeps every host CPU for the cpu_baseline leg
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    est = make_estimator()
    nb = 4
    batches = host_batches(nb, seed0=1234 + 100 * rank)
    dev_batches = [est.to_device(b) for b in batches]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def step_resident(i):
        return est.predict_device(dev_batches[i % nb])     # the PREDICT path of Estimator.predict*, inputs resident

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also builds variables / packs weights)
    for i in range(max(args.warmup, 3)):
        step_resident(i)
    barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- device-resident timing: K steps, L2 flushed (untimed) between steps
    evs = []
    barrier()
    l0 = _lib.LAUNCHES
    for i in range(args.steps):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        last_pred = step_resident(i)
        e.record()
        evs.append((s, e))
    barrier()
    # --dump-outputs: this loop's last step, and below the last batch of every timed pipeline configuration (each one, not
    # only the one that sets `value`: that choice is made by timing, the set of configurations by the arguments)
    outputs = {"pred_ids": last_pred.cpu().numpy()}
    launches = _lib.LAUNCHES - l0
    t_res = sum(s.elapsed_time(e) for s, e in evs) / 1e3

    # ---- the same K steps as a throughput pipeline (sentences are independent, SURVEY 8(e)):
    #      * NS CUDA streams: consecutive calls alternate over streams, so the SMs one call's kernel leaves idle in its
    #        partial last wave run another call's kernels;
    #      * G batches stacked per call: the packed token count of one 64-sentence MSRA batch (~3.2 k rows) is 0.5 / 1.5 /
    #        2.0 waves of 128x256 tiles on 148 SMs, two batches are 1.0 / 3.0 / 4.0.
    #      One event pair around the K steps; no flush kernel (the 170 MB of bf16 weights streamed per call exceed the
    #      126 MB L2).  Every combination processes the same K batches; the best one is the line's `value`.
    from chinesener_b200 import ops as _ops
    stacked = {1: dev_batches}

    def dev_group(G):
        if G not in stacked:
            stacked[G] = [est.stack_to_device([batches[(j * G + q) % nb] for q in range(G)]) for j in range(max(1, nb // G))]
            torch.cuda.synchronize()
        return stacked[G]

    def time_pipeline(NS, G):
        groups = dev_group(G)
        calls = [(j, min(G, args.steps - j * G)) for j in range((args.steps + G - 1) // G)]     # (call index, batches in it)
        for _, nbat in calls:
            dev_group(nbat)                            # stacked inputs of a short last call are built outside the timed region
        assert sum(n for _, n in calls) == args.steps
        side = [torch.cuda.Stream() for _ in range(NS)]
        _ops.DEFAULT_TILE = _ops.TILE_AUTO_THROUGHPUT   # partial waves are filled by other streams / stacked rows: fastest tile
        try:
            def run(j, nbat):
                grp = groups if nbat == G else dev_group(nbat)      # the last call of the K steps may hold fewer batches
                with torch.cuda.stream(side[j % NS]):
                    return est.predict_device(grp[j % len(grp)])
            for j in range(2 * NS):
                run(j, G)
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for st in side:
                st.wait_event(s)
            for j, nbat in calls:
                last_pred = run(j, nbat)
            for st in side:
                torch.cuda.current_stream().wait_stream(st)
            e.record()
            barrier()
        finally:
            _ops.DEFAULT_TILE = 0
        return s.elapsed_time(e) / 1e3, last_pred[-B_PER_GPU:].cpu().numpy()     # the last call's last 64-sentence batch

    combos = [(max(2, args.streams), 1), (max(1, args.group_streams), max(1, args.group))]
    if args.sweep:
        combos = sorted(set(combos + [(1, 2), (2, 2), (3, 2), (1, 4), (2, 4), (3, 4), (4, 4), (2, 6), (2, 8), (3, 8), (2, 1), (3, 1)]))
    pipe = {}
    for NS_, G_ in combos:
        t, outputs[f"pred_ids_pipeline_streams{NS_}_batches{G_}"] = time_pipeline(NS_, G_)
        if dist is not None:                        # max over ranks decides, every rank must pick the same combination
            tt = torch.tensor([t], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_all = float(tt[0])
        else:
            t_all = t
        pipe[(NS_, G_)] = (t, t_all)
    (NS, G) = min(pipe, key=lambda k: pipe[k][1])
    t_res2 = pipe[(NS, G)][0]

    # ---- end-to-end timing through the public PREDICT API, Estimator.predict_iter (the generator shape of
    #      tf.estimator.Estimator.predict): every step copies its pinned host batch H2D and its pred_ids D2H inside
    #      the timed region; the next call is enqueued while the previous result is awaited.  One event pair around
    #      the K steps (per-step brackets do not exist in a pipelined loop); no flush kernel here: the 170 MB of
    #      bf16 weights streamed every call already exceed the 126 MB L2.  Same (streams, batches per call) as `value`.
    #      The API's own pipeline parameters are chosen the same way as for `value`: the two best resident combinations are
    #      timed end to end and the better one is reported (a deep stack pays a longer fill / drain over only K = 20 steps).
    def time_e2e(ns_, g_):
        for _ in est.predict_iter((batches[i % nb] for i in range(2 * ns_ * g_)), depth=ns_ + 1, streams=ns_, group=g_):
            pass
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        n_out = 0
        for out in est.predict_iter((batches[i % nb] for i in range(args.steps)), depth=ns_ + 1, streams=ns_, group=g_):
            n_out += out['pred_ids'].shape[0]
        e.record()
        barrier()
        assert n_out == B_PER_GPU * args.steps
        t = s.elapsed_time(e) / 1e3
        if dist is not None:
            tt = torch.tensor([t], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return t, float(tt[0])
        return t, t

    e2e_all = {}
    for k in sorted(pipe, key=lambda k: pipe[k][1])[:2]:
        e2e_all[k] = time_e2e(*k)
    (NS_E, G_E) = min(e2e_all, key=lambda k: e2e_all[k][1])
    t_e2e = e2e_all[(NS_E, G_E)][0]
    # unpipelined variant (one blocking Estimator.predict per batch), reported beside it
    evs = []
    for i in range(args.steps):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = est.predict(batches[i % nb])  # .cpu() inside synchronises on the result
        e.record()
        evs.append((s, e))
    barrier()
    t_e2e_blocking = sum(s.elapsed_time(e) for s, e in evs) / 1e3

    # ---- TRAIN step (SURVEY 8(d)(i) second figure): forward with the tape + backward + the data-parallel gradient
    #      exchange (N>1: bucketed all-reduces overlapped with the backward pass) + AdamW, device-resident batches
    t_train, train_extra = None, {}

    def time_train(est_t, dev_list, steps):
        evs = []
        barrier()
        for i in range(steps):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            est_t.train_step(dev_list[i % len(dev_list)])
            e.record()
            evs.append((s, e))
        barrier()
        return sum(s.elapsed_time(e) for s, e in evs) / 1e3

    def max_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt[0])

    if not args.no_train:
        est_t = make_estimator()
        est_t.params.update(num_train_steps=10000, warmup_ratio=0.1)
        for i in range(3):
            est_t.train_step(dev_batches[i % nb])
        t_train = time_train(est_t, dev_batches, args.steps)
        if dist is not None:
            # the exchange's share: the same step with ONE all-reduce after the backward pass (round-1 behaviour), with the
            # bf16 buckets, and with no exchange at all (diagnostic: what perfect overlap would read)
            k2 = min(args.steps, 10)
            for mode in ("single", "overlap_bf16", "skip"):
                est_t.store.grad_exchange = mode
                est_t.store._grad_exchange = None
                est_t.train_step(dev_batches[0])
                train_extra[mode + "_ms_per_step"] = 1e3 * max_over_ranks(time_train(est_t, dev_batches, k2)) / k2
            est_t.store.grad_exchange = "overlap"
            est_t.store._grad_exchange = None
            # strong scaling (SURVEY 8e "Reporting"): the global batch stays 64, every rank steps over 64 / N sentences
            Bs = max(B_PER_GPU // world, 1)
            small = [est.to_device({k: (v[rank * Bs % B_PER_GPU: rank * Bs % B_PER_GPU + Bs] if torch.is_tensor(v) else v) for k, v in b.items()})
                     for b in batches]
            est_t.train_step(small[0])
            k2 = min(args.steps, 10)
            t_strong_train = max_over_ranks(time_train(est_t, small, k2)) / k2
            for i in range(3):
                est.predict_device(small[i % nb])
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(args.steps):
                est.predict_device(small[i % nb])
            e.record()
            barrier()
            t_strong_pred = max_over_ranks(s.elapsed_time(e) / 1e3) / args.steps
            train_extra["strong_scaling"] = {"global_batch": Bs * world, "per_gpu_batch": Bs,
                                             "train_ms_per_step": 1e3 * t_strong_train, "train_sentences_per_sec": Bs * world / t_strong_train,
                                             "predict_ms_per_step": 1e3 * t_strong_pred, "predict_sentences_per_sec": Bs * world / t_strong_pred,
                                             "note": "global batch fixed at 64 sentences: per-GPU work shrinks with N (latency / exchange bound)"}
        del est_t

    # ---- host enqueue time of one step (GPU parked behind a spin kernel): says whether the step is launch-bound
    torch.cuda.synchronize()
    torch.cuda._sleep(40_000_000)
    h0 = time.perf_counter()
    for i in range(5):
        step_resident(i)
    host_ms = (time.perf_counter() - h0) * 1e3 / 5
    torch.cuda.synchronize()

    per_rank = None
    if dist is not None:
        mine = torch.tensor([t_res, t_res2, t_e2e, t_train or 0.0, host_ms], device="cuda", dtype=torch.float64)
        allr = torch.empty((world, mine.numel()), device="cuda", dtype=torch.float64)
        dist.all_gather_into_tensor(allr, mine)
        per_rank = {"columns": ["single_stream_s", "multi_stream_s", "e2e_s", "train_s", "host_enqueue_ms_per_step"],
                    "rows": [[round(float(x), 6) for x in r] for r in allr.cpu()]}
        t = torch.tensor([t_res, t_e2e, t_train or 0.0, t_res2], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_res, t_e2e, t_res2 = float(t[0]), float(t[1]), float(t[3])
        t_train = float(t[2]) if t_train is not None else None

    # ---- roofline of the dominant kernel (tcgen05 GEMM), instrumented pass on rank 0
    roof = cpu = None
    if rank == 0:
        hbm_peak, tf_peak, how = measured_peaks()
        from chinesener_b200 import bert as _bert
        timer = GemmTimer()
        _lib._HOOK = timer
        _bert.PER_KERNEL = True          # same kernels, one C-ABI call each, so every GEMM launch gets its own events
        _ops.DEFAULT_TILE = _ops.TILE_AUTO_THROUGHPUT if t_res2 <= t_res else 0      # the tile policy of the selected pipeline
        n_roof = min(args.steps, 5)
        for i in range(n_roof):
            # per-kernel calls come from Python (~20 us of host time each): hold the GPU behind a spin kernel so the
            # whole call is enqueued first and the event pairs bracket execution, not launch latency
            torch.cuda._sleep(20_000_000 * (G if t_res2 <= t_res else 1))
            est.predict_device(dev_group(G)[i % len(dev_group(G))] if t_res2 <= t_res else dev_batches[i % nb])
            torch.cuda.synchronize()
        _ops.DEFAULT_TILE = 0
        _bert.PER_KERNEL = False
        _lib._HOOK = None
        ms, fl, n = timer.summary()
        achieved = fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        roof = {"bound": "tensor", "kernel": "gemm_bf16_tc_kernel (tcgen05.mma kind::f16, all dense layers)",
                "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                # DRAM bytes per launch are not measurable inside an un-profiled run; the `ncu --set full` capture of an
                # in-step launch lives in profiles/ (README there) and is quoted in DESIGN.md, not here
                "traffic": None,
                "peak_source": f"{how} bf16_tflops_sustained", "launches_timed": n,
                "batches_per_timed_call": G if t_res2 <= t_res else 1,
                "gemm_share_of_step": ((ms / n_roof / (G if t_res2 <= t_res else 1)) / (1e3 * t_res / args.steps) if t_res > 0 else None),
                "gemm_share_note": "GEMM ms per 64-sentence batch (from the timed calls) / single-stream single-batch ms per step"}
        extra = {}
        if not args.no_kernel_rooflines and world == 1:     # single-GPU kernel figures: reported on the N=1 line
            extra.update(crf_rooflines(hbm_peak, f"{how} hbm_gbs"))
            extra["roofline_softlexicon"] = softlexicon_roofline(hbm_peak, f"{how} hbm_gbs", flush)
            extra["configs"] = other_configs(min(args.steps, 20), flush)
        clocks = sampler.stop()        # the NVML record covers every GPU-timed region above; the CPU leg below is host-only
        if world == 1 and not args.no_cpu_baseline:
            from chinesener_b200 import synthetic as _syn
            oparams = dict(_syn.data_params(SEQ_LEN, LABELS), rnn_activation=est.params['rnn_activation'])
            hb = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in b.items()} for b in batches[:2]]
            v, ts, first = time_cpu_reference(est.store.state_dict(), oparams, hb, reps=2)
            cpu = {"value": v, "unit": "sentences/sec", "cores": pick_cpu_threads(), "host_cpus": os.cpu_count(), "kind": "port",
                   "sample": f"2 timed reps x one 64-sentence batch (L=128) of the timed workload, same weights as the GPU arm; "
                             f"PyTorch-CPU fp32 restatement of model/bert_bilstm_crf.py (TF 1.14 not installable); rep seconds "
                             f"{['%.2f' % x for x in ts]}"}
            extra["parity"] = check_parity(est, batches[0], first)
            extra["parity_checked"] = extra["parity"]["parity_checked"]
        else:
            extra["parity_checked"] = False

    if rank == 0:
        sent = B_PER_GPU * world * args.steps
        t_best = min(t_res, t_res2)
        h2d = sum(v.numel() * v.element_size() for v in batches[0].values())
        d2h = B_PER_GPU * SEQ_LEN * 4
        line = {
            "metric": METRIC, "value": sent / t_best, "unit": "sentences/sec", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * t_best / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": B_PER_GPU * world, "seq_len": SEQ_LEN,
                       "parallelism": f"dp{world} (sentence-sharded, no data-path collective in PREDICT)",
                       "l2": "working set/step > 126 MB L2 (170 MB bf16 weights + activations); L2 also flushed by an "
                             "untimed 256 MB write between timed steps",
                       "lengths": "MSRA-shaped (mean fill ~0.39)",
                       "streams": (f"{NS} CUDA stream(s) per GPU, consecutive calls alternate; {G} batch(es) of 64 sentences stacked per "
                                   f"call" if t_res2 <= t_res else "1 stream, 1 batch per call"),
                       "single_stream_ms_per_step": 1e3 * t_res / args.steps,
                       "pipeline_ms_per_step": {f"streams={k[0]},batches_per_call={k[1]}": 1e3 * v[1] / args.steps for k, v in pipe.items()}},
            "e2e": {"value": sent / t_e2e, "unit": "sentences/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * t_e2e / args.steps, "api": f"Estimator.predict_iter(depth={NS_E + 1}, streams={NS_E}, group={G_E})",
                    "candidates_ms_per_step": {f"streams={k[0]},group={k[1]}": 1e3 * v[1] / args.steps for k, v in e2e_all.items()},
                    "blocking_predict_ms_per_step": 1e3 * t_e2e_blocking / args.steps},
            "gpu_launches": launches, "host_enqueue_ms_per_step": host_ms, "clocks": clocks, "roofline": roof,
            "per_rank": per_rank, "cpu_affinity": numa,
        }
        if t_train is not None:
            line["train"] = {"value": sent / t_train, "unit": "sentences/sec", "ms_per_step": 1e3 * t_train / args.steps,
                             "what": "TRAIN step of the same plugin: forward (sequence-packed encoder, dropout on) + backward + "
                                     + ("bucketed NCCL all-reduces of the flat fp32 gradient buffer overlapped with the backward pass + " if world > 1 else "")
                                     + "global-norm clip + AdamW (bert_train_op); device-resident batches"}
        if t_train is not None and train_extra:
            line["train"]["exchange"] = train_extra
        if cpu is not None:
            line["cpu_baseline"] = cpu
        line.update(extra)
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-kernel-rooflines", dest="no_kernel_rooflines", action="store_true",
                    help="skip the stand-alone CRF / SoftLexicon roofline runs and the config 2/4/5 PREDICT timings")
    ap.add_argument("--no-train", dest="no_train", action="store_true", help="skip the TRAIN-step figure")
    ap.add_argument("--streams", type=int, default=4, help="CUDA streams per GPU that consecutive single-batch PREDICT calls alternate over")
    ap.add_argument("--group", type=int, default=4, help="batches stacked per PREDICT call in the second pipeline configuration")
    ap.add_argument("--group-streams", dest="group_streams", type=int, default=2, help="CUDA streams of the stacked configuration")
    ap.add_argument("--sweep", action="store_true", help="time more (streams, batches per call) combinations")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the pred_ids [64, 128] of the last timed step (rank 0) to DIR/pred_ids.npy, "
                         "and those of the last batch of each timed pipeline configuration to DIR/pred_ids_pipeline_*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
