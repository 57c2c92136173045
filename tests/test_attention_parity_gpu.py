"""GPU: every dispatch path of the BERT attention core against the float64 reference of _attention_ref.py, per (sequence,
head) block under the bound err <= TAU * rms + 2^-9 * max|X64|:
  fwd_tc        the default inference forward (tcgen05, attention_tc.cu; keys <= 256)
  fwd_mma       NER_ATTN_VARIANT=1, the mma.sync forward (attention.cu), keys up to 768
  fwd_mma_drop  keep_prob 0.9: the mma.sync forward with attention-probs dropout
  bwd/bwd_drop  attention_bwd.cu, padded and packed, keep_prob 1.0 / 0.9, keys up to 384
plus hostile neighbours, head isolation, the length limits and the QKV alignment check.  test_attention_reference.py shows
on the CPU that the bound holds the kernels' bf16 rounding with a factor-3 margin and that each of a set of plausible
indexing / scaling / dropout bugs would break it."""
import subprocess

import pytest
import torch

import _attention_ref as R
from chinesener_b200 import ops
from chinesener_b200._lib import NerB200Error

pytestmark = pytest.mark.gpu
D = R.D
WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    print(f"\n{torch.cuda.get_device_name()}, power limit {power}: worst err/bound per path")
    for path, (ratio, where) in sorted(WORST.items()):
        print(f"  {path:13s} {ratio:.3f}  ({where})")


def _run(case, path, qkv, dout, monkeypatch):
    """the kernel's output parts as float64 [T, NH, D]"""
    direction, keep, variant = R.PATHS[path]
    if variant is not None:
        monkeypatch.setenv("NER_ATTN_VARIANT", variant)
    else:
        monkeypatch.delenv("NER_ATTN_VARIANT", raising=False)
    packed = case.layout == "packed"
    mask = None if packed else case.mask.cuda()
    cu = torch.tensor(case.cu, dtype=torch.int32).cuda() if packed else None
    kw = dict(scale=case.scale, cu_seqlens=cu, keep_prob=keep, seed=R.SEED)
    if direction == "fwd":
        out = ops.bert_attention(qkv.cuda(), mask, case.B, case.L, case.NH, D, **kw)
        return {"o": out.cpu().double().reshape(case.T, case.NH, D)}
    ctx = R.ctx_for_bwd(case, qkv, keep).cuda()
    g = ops.bert_attention_bwd(qkv.cuda(), mask, ctx, dout.cuda(), case.B, case.L, case.NH, D, **kw)
    g = g.cpu().double().reshape(case.T, 3, case.NH, D)
    return {"dq": g[:, 0], "dk": g[:, 1], "dv": g[:, 2]}


CASES = [(path, c) for path in R.PATHS for c in R.cases_for(path)]


@pytest.mark.parametrize("path,case", CASES, ids=[f"{p}-{c.name}" for p, c in CASES])
def test_matches_float64_reference(path, case, monkeypatch):
    qkv, dout = R.make_inputs(case)
    outs = _run(case, path, qkv, dout, monkeypatch)
    ratio, where = R.worst_ratio(case, outs, R.reference(case, path, qkv, dout), path)
    if ratio >= WORST.get(path, (-1.0, None))[0]:
        WORST[path] = (ratio, f"{case.name}, part {where[0]}, seq/len/head {where[1]}")
    print(f"{path} {case.name}: worst err/bound {ratio:.3f} at {where}")
    assert ratio <= 1.0, (ratio, where)


# --------------------------------------------------------------------------- hostile neighbours, head isolation
def _poison_rows(t, rows, cols):
    t = t.clone()
    half = rows.start + (rows.stop - rows.start) // 2
    t[rows.start:half, cols] = float("inf")
    t[half:rows.stop, cols] = float("nan")
    return t


@pytest.mark.parametrize("keep", [1.0, 0.9])
def test_mma_forward_ignores_hostile_neighbours(keep, monkeypatch):
    """sequence 0 is short; sequence 1's K is huge, its Q / V are inf / NaN: sequence 0's context must be bit-identical to
    its stand-alone result and finite"""
    monkeypatch.setenv("NER_ATTN_VARIANT", "1")
    NH, lens = 2, [19, 90]
    qkv = R.make_inputs(R.Case("n", NH, lens=lens, seed=21))[0]
    alone = ops.bert_attention(qkv[:19].contiguous().cuda(), None, 1, 19, NH, D, keep_prob=keep, seed=5,
                               cu_seqlens=torch.tensor([0, 19], dtype=torch.int32).cuda())
    bad = qkv.clone()
    bad[19:, NH * D:2 * NH * D] = 3.0e4
    bad = _poison_rows(bad, slice(19, 109), slice(0, NH * D))
    bad = _poison_rows(bad, slice(19, 109), slice(2 * NH * D, 3 * NH * D))
    out = ops.bert_attention(bad.cuda(), None, 2, 90, NH, D, keep_prob=keep, seed=5,
                             cu_seqlens=torch.tensor([0, 19, 109], dtype=torch.int32).cuda())
    assert torch.equal(out[:19], alone)
    assert torch.isfinite(out[:19].float()).all()


@pytest.mark.parametrize("keep", [1.0, 0.9])
def test_packed_backward_ignores_hostile_neighbours(keep):
    """as above for ner_bert_attention_bwd_packed: the neighbour's K is huge, its Q / V / dO / ctx are inf / NaN"""
    NH, lens = 2, [19, 90]
    case = R.Case("n", NH, lens=lens, seed=22)
    qkv, dout = R.make_inputs(case)
    ctx = R.ctx_for_bwd(case, qkv, keep)
    one = torch.tensor([0, 19], dtype=torch.int32).cuda()
    alone = ops.bert_attention_bwd(qkv[:19].contiguous().cuda(), None, ctx[:19].contiguous().cuda(),
                                   dout[:19].contiguous().cuda(), 1, 19, NH, D, keep_prob=keep, seed=5, cu_seqlens=one)
    bad = qkv.clone()
    bad[19:, NH * D:2 * NH * D] = 3.0e4
    bad = _poison_rows(bad, slice(19, 109), slice(0, NH * D))
    bad = _poison_rows(bad, slice(19, 109), slice(2 * NH * D, 3 * NH * D))
    bad_ctx = _poison_rows(ctx, slice(19, 109), slice(0, NH * D))
    bad_dout = _poison_rows(dout, slice(19, 109), slice(0, NH * D))
    g = ops.bert_attention_bwd(bad.cuda(), None, bad_ctx.cuda(), bad_dout.cuda(), 2, 90, NH, D, keep_prob=keep, seed=5,
                               cu_seqlens=torch.tensor([0, 19, 109], dtype=torch.int32).cuda())
    assert torch.equal(g[:19], alone)
    assert torch.isfinite(g[:19].float()).all()


def _head_cols(NH, h, parts):
    return torch.cat([torch.arange(D) + (p * NH + h) * D for p in range(parts)])


@pytest.mark.parametrize("path", ["fwd_tc", "fwd_mma", "bwd"])
def test_heads_are_isolated(path, monkeypatch):
    """every other head's Q / K / V (and ctx / dO) columns are NaN: head h's result equals its stand-alone NH = 1 result"""
    NH, lens = 3, [70, 130, 5]
    case = R.Case("iso", NH, lens=lens, styles=R.MIX, seed=23)
    qkv, dout = R.make_inputs(case)
    ctx = R.ctx_for_bwd(case, qkv, 1.0)
    cu = torch.tensor(case.cu, dtype=torch.int32).cuda()
    if path == "fwd_mma":
        monkeypatch.setenv("NER_ATTN_VARIANT", "1")
    else:
        monkeypatch.delenv("NER_ATTN_VARIANT", raising=False)
    for h in range(NH):
        qc, oc = _head_cols(NH, h, 3), _head_cols(NH, h, 1)
        bad_qkv = torch.full_like(qkv, float("nan"))
        bad_qkv[:, qc] = qkv[:, qc]
        if path.startswith("fwd"):
            alone = ops.bert_attention(qkv[:, qc].contiguous().cuda(), None, 3, 130, 1, D, cu_seqlens=cu)
            out = ops.bert_attention(bad_qkv.cuda(), None, 3, 130, NH, D, cu_seqlens=cu)
            assert torch.equal(out[:, oc], alone), h
        else:
            bad_ctx, bad_dout = torch.full_like(ctx, float("nan")), torch.full_like(dout, float("nan"))
            bad_ctx[:, oc], bad_dout[:, oc] = ctx[:, oc], dout[:, oc]
            alone = ops.bert_attention_bwd(qkv[:, qc].contiguous().cuda(), None, ctx[:, oc].contiguous().cuda(),
                                           dout[:, oc].contiguous().cuda(), 3, 130, 1, D, cu_seqlens=cu)
            g = ops.bert_attention_bwd(bad_qkv.cuda(), None, bad_ctx.cuda(), bad_dout.cuda(), 3, 130, NH, D, cu_seqlens=cu)
            assert torch.equal(g[:, qc], alone), h
        assert torch.isfinite(alone.float()).all()


# --------------------------------------------------------------------------- loud limits, alignment
@pytest.mark.parametrize("keep", [1.0, 0.9])
@pytest.mark.parametrize("packed", [False, True])
def test_forward_length_limit(packed, keep):
    """L = 768 runs (the reference cases cover its values); L = 769 is refused before any launch"""
    for L, ok in ((768, True), (769, False)):
        qkv = torch.zeros(L, 3 * D, dtype=torch.bfloat16, device="cuda")
        mask = None if packed else torch.ones(1, L, dtype=torch.int32, device="cuda")
        cu = torch.tensor([0, L], dtype=torch.int32, device="cuda") if packed else None
        if ok:
            out = ops.bert_attention(qkv, mask, 1, L, 1, D, cu_seqlens=cu, keep_prob=keep)
            torch.cuda.synchronize()
            assert torch.isfinite(out.float()).all()
        else:
            with pytest.raises(NerB200Error):
                ops.bert_attention(qkv, mask, 1, L, 1, D, cu_seqlens=cu, keep_prob=keep)


@pytest.mark.parametrize("packed", [False, True])
def test_backward_length_limit(packed):
    """L = 384 runs; L = 385 is refused before any launch"""
    for L, ok in ((384, True), (385, False)):
        qkv = torch.zeros(L, 3 * D, dtype=torch.bfloat16, device="cuda")
        ctx, dout = (torch.zeros(L, D, dtype=torch.bfloat16, device="cuda") for _ in range(2))
        mask = None if packed else torch.ones(1, L, dtype=torch.int32, device="cuda")
        cu = torch.tensor([0, L], dtype=torch.int32, device="cuda") if packed else None
        if ok:
            g = ops.bert_attention_bwd(qkv, mask, ctx, dout, 1, L, 1, D, cu_seqlens=cu)
            torch.cuda.synchronize()
            assert float(g.float().abs().max()) == 0.0
        else:
            with pytest.raises(NerB200Error):
                ops.bert_attention_bwd(qkv, mask, ctx, dout, 1, L, 1, D, cu_seqlens=cu)


def _misaligned(rows, cols):
    """a contiguous bf16 [rows, cols] view whose first element sits 2 bytes past a 16-byte boundary"""
    buf = torch.zeros(rows * cols + 8, dtype=torch.bfloat16, device="cuda")
    t = buf[1:1 + rows * cols].view(rows, cols)
    assert t.is_contiguous() and t.data_ptr() % 16 == 2
    return t


def _require_library_from_this_tree():
    """A library built before the alignment check would hand these views to 16-byte cp.async copies and fault, taking
    the CUDA context down with it.  So nothing misaligned is passed unless the loaded libner_b200.so was built from the
    sources of this tree (ner_build_info() echoes the source hash it was compiled from)."""
    from chinesener_b200 import build
    from chinesener_b200._lib import lib
    want = "src=" + build.source_hash()
    if want not in lib().ner_build_info().decode():
        pytest.fail(f"libner_b200.so was not built from this tree ({want} missing): run python -m chinesener_b200.build")


@pytest.mark.parametrize("variant", [None, "1"])
@pytest.mark.parametrize("keep", [1.0, 0.9])
def test_misaligned_qkv_is_refused(variant, keep, monkeypatch):
    _require_library_from_this_tree()
    if variant is None:
        monkeypatch.delenv("NER_ATTN_VARIANT", raising=False)
    else:
        monkeypatch.setenv("NER_ATTN_VARIANT", variant)
    L, NH = 40, 2
    cu = torch.tensor([0, L], dtype=torch.int32, device="cuda")
    mask = torch.ones(1, L, dtype=torch.int32, device="cuda")
    for m, c in ((mask, None), (None, cu)):
        with pytest.raises(NerB200Error):
            ops.bert_attention(_misaligned(L, 3 * NH * D), m, 1, L, NH, D, cu_seqlens=c, keep_prob=keep)
    ok = lambda rows, cols: torch.zeros(rows, cols, dtype=torch.bfloat16, device="cuda")
    for m, c in ((mask, None), (None, cu)):
        for bad in range(3):
            args = [ok(L, 3 * NH * D), ok(L, NH * D), ok(L, NH * D)]
            args[bad] = _misaligned(*args[bad].shape)
            with pytest.raises(NerB200Error):
                ops.bert_attention_bwd(args[0], m, args[1], args[2], 1, L, NH, D, cu_seqlens=c, keep_prob=keep)
    torch.cuda.synchronize()
