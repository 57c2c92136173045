"""CPU: the float64 attention reference of _attention_ref.py is self-consistent, the committed tolerances TAU hold the bf16
emulation of each kernel path with a factor-3 margin on the inputs the GPU tests use, and every deliberately wrong reference
lands at least 3x outside the bound on at least one of those inputs -- so test_attention_parity_gpu.py can fail."""
import functools
import math

import numpy as np
import pytest
import torch

import _attention_ref as R
from _masks import attention_keep


@functools.lru_cache(maxsize=None)
def _inputs(name, path):
    case = next(c for c in R.cases_for(path) if c.name == name)
    qkv, dout = R.make_inputs(case)
    return case, qkv, dout


@functools.lru_cache(maxsize=None)
def _refs(name, path):
    case, qkv, dout = _inputs(name, path)
    return R.reference(case, path, qkv, dout)


def _cost(case):
    return case.NH * (sum(n * n for n in case.lens) if case.layout == "packed" else case.B * case.L * case.L)


def test_keep_z_matches_the_mask_helper():
    B, NH, L, seed = 3, 2, 70, 0x5EED_0000_0077
    full = attention_keep(B, NH, L, 0.9, seed)
    for b in range(B):
        z = R.keep_z(b, NH, L, L, 0.9, seed)
        assert np.array_equal(z.numpy() > 0, full[b])
        assert float(z.max()) == float(np.float32(1) / np.float32(0.9))


@pytest.mark.parametrize("keep", [1.0, 0.9])
def test_packed_reference_equals_padded_on_real_rows(keep):
    lens = [7, 64, 1, 130, 65]
    L, NH = max(lens), 2
    padded = R.Case("p", NH, mask=(torch.arange(L)[None, :] < torch.tensor(lens)[:, None]).int(), styles=R.MIX, seed=1)
    packed = R.Case("q", NH, lens=lens, styles=R.MIX, seed=1)
    qkv_pad, dout_pad = R.make_inputs(padded)
    real = torch.cat([torch.arange(n) + b * L for b, n in enumerate(lens)])
    qkv, dout = qkv_pad[real], dout_pad[real]
    o_pad = R.forward(padded, qkv_pad, keep)[real]
    o = R.forward(packed, qkv, keep)
    assert float((o - o_pad).abs().max()) < 1e-12
    pad_rows_silent = torch.zeros(padded.T, 1, dtype=torch.bfloat16)   # [PAD] queries would reach real keys in padded mode
    pad_rows_silent[real] = 1
    g_pad = R.backward(padded, qkv_pad, dout_pad * pad_rows_silent, keep)
    g = R.backward(packed, qkv, dout, keep)
    for a, b_ in zip(g, g_pad):
        assert float((a - b_[real]).abs().max()) < 1e-10


@pytest.mark.parametrize("keep", [1.0, 0.9])
@pytest.mark.parametrize("layout", ["packed", "padded"])
def test_autograd_equals_the_closed_form(layout, keep):
    if layout == "packed":
        case = R.Case("c", 3, lens=[1, 40, 0, 77], styles=("random", "peaked", "sink"), seed=5)
    else:
        case = R.Case("c", 2, mask=R._holes_mask(3, 50, 5), styles=R.MIX, seed=5)
    qkv, dout = R.make_inputs(case)
    dq, dk, dv, o = R.backward(case, qkv, dout, keep)
    cq, ck, cv = R.backward_closed(case, qkv, dout, keep)
    for a, b_ in ((dq, cq), (dk, ck), (dv, cv)):
        assert float((a - b_).abs().max()) <= 1e-10 * max(1.0, float(b_.abs().max()))
    assert float((o - R.forward(case, qkv, keep)).abs().max()) == 0.0


def test_emulations_are_exact_when_nothing_rounds():
    """sanity of the emulations themselves: at one key per sequence every probability is exactly 1 and ctx = v"""
    case = R.Case("one", 2, lens=[1, 1, 1], seed=3)
    qkv, dout = R.make_inputs(case)
    v = qkv.double().reshape(3, 3, 2, R.D)[:, 2]
    assert torch.equal(R.emulate_fwd_tc(case, qkv), v)
    assert torch.equal(R.emulate_fwd_mma(case, qkv), v)


@pytest.mark.parametrize("path", list(R.PATHS))
def test_tau_holds_the_bf16_emulation_with_margin_3(path):
    worst = {}
    for case in R.cases_for(path):
        _, qkv, dout = _inputs(case.name, path)
        need = R.needed_tau(case, R.emulation(case, path, qkv, dout), _refs(case.name, path))
        for part, t in need.items():
            if t >= worst.get(part, (-1.0, None))[0]:
                worst[part] = (t, case.name)
    print()
    for part, (t, name) in worst.items():
        print(f"{path:13s} {part}: emulation needs tau {t:.4f} ({name}); 3x = {3 * t:.4f} <= TAU {R.TAU[(path, part)]}")
    assert all(3.0 * t <= R.TAU[(path, part)] for part, (t, _) in worst.items())


@pytest.mark.parametrize("path", list(R.PATHS))
def test_every_mutation_reaches_3x_the_bound(path):
    """each wrong reference must miss the float64 one by >= 3 bounds on some case of the path; cases are tried cheapest
    first and the two first that catch a mutation are printed"""
    print()
    cases = sorted(R.cases_for(path), key=_cost)
    for mut in R.mutations_for(path):
        caught = []
        for case in cases:
            if not R.applies(case, mut):
                continue
            _, qkv, dout = _inputs(case.name, path)
            ratio, where = R.worst_ratio(case, R.mutated(case, path, qkv, dout, mut), _refs(case.name, path), path)
            if ratio >= 3.0:
                caught.append(f"{case.name} ({ratio:.3g}x at {where[0]} seq/len/head {where[1]})")
                if len(caught) == 2:
                    break
        print(f"{path:13s} {mut:15s} caught by: {'; '.join(caught) if caught else 'NOTHING'}")
        assert caught, (path, mut)


def test_bound_is_per_block():
    """the bound is judged per (sequence, head) block and names the block that fails; NaN never passes"""
    case = R.Case("c", 1, lens=[3, 4, 5, 200], seed=9)
    qkv, _ = R.make_inputs(case)
    ref = R.forward(case, qkv)
    bad = ref.clone()
    bad[12:] *= 1.05
    ratio, where = R.worst_ratio(case, {"o": bad}, {"o": ref}, "fwd_tc")
    assert ratio > 1.0 and where[1][0] == 3
    assert R.worst_ratio(case, {"o": ref}, {"o": ref}, "fwd_tc")[0] == 0.0
    nan = ref.clone()
    nan[0, 0, 0] = math.nan
    assert R.worst_ratio(case, {"o": nan}, {"o": ref}, "fwd_tc")[0] == math.inf
