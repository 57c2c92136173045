"""float64 reference of the BERT self-attention core (csrc/attention.cu, attention_tc.cu, attention_bwd.cu), rounding-point
emulations of the three kernels, deliberately wrong ("mutated") references, the error bound the GPU tests apply, and the
test cases they run.  Everything is computed on the CPU from the same bf16 inputs a kernel gets.

Layouts.  Padded: qkv [B*L, 3*NH*64], sequence b owns rows [b*L, (b+1)*L), key k gets the additive (1 - mask[b, k]) * mask_add
and every row is a query.  Packed: qkv [T, 3*NH*64], sequence b owns rows [cu[b], cu[b+1]), every key is valid.  Dropout of
the attention probabilities uses z(b, h, q, k) = keep(b, h, q, k) / keep_prob with local query / key indices in both layouts
(the kernels' counter hash, restated in _masks.py).

Bound.  For each output part X (ctx; or dQ, dK, dV) and each (sequence, head) block over the sequence's rows:
    err = max |X - X64|,   bound = tau[path, part] * rms(X64 on the block) + 2^-9 * max |X64|,
where the max in the floor runs over the same block, so a large block elsewhere in the batch loosens no other block's
bound (over all three parts of the block when the part is identically zero there, as dQ and dK are for a one-key
sequence).  tau is fixed in TAU; test_attention_reference.py checks that it is at
least 3x what the bf16 emulation of the path needs on the very inputs the GPU tests use, and that every mutation reaches
3x the bound on at least one of them."""
import math

import numpy as np
import torch

from _masks import hash3, keep_threshold

D = 64
MASK_ADD = -10000.0
LOG2E = 1.4426950408889634
FLOOR = 2.0 ** -9

# committed tolerances per (path, part).  Derivation: 3 x the largest tau the bf16 emulation of the path needs over all
# its cases (printed by test_tau_holds_the_bf16_emulation_with_margin_3; 3x need in the comments), rounded up by ~5-10 %.
# Adding or reseeding a case can raise the need: rerun that test and, if it fails, raise tau only as far as the new 3x
# need -- and then check that test_every_mutation_reaches_3x_the_bound still passes.
TAU = {
    ("fwd_tc", "o"): 0.035,                # 3x need 0.0328
    ("fwd_mma", "o"): 0.035,               # 0.0328
    ("fwd_mma_drop", "o"): 0.06,           # 0.0546
    ("bwd", "dq"): 0.14,                   # 0.1325
    ("bwd", "dk"): 0.12,                   # 0.1110
    ("bwd", "dv"): 0.065,                  # 0.0591
    ("bwd_drop", "dq"): 0.125,             # 0.1156
    ("bwd_drop", "dk"): 0.135,             # 0.1241
    ("bwd_drop", "dv"): 0.09,              # 0.0810
}
PATHS = {  # path -> (direction, keep_prob, NER_ATTN_VARIANT)
    "fwd_tc": ("fwd", 1.0, None),
    "fwd_mma": ("fwd", 1.0, "1"),
    "fwd_mma_drop": ("fwd", 0.9, None),
    "bwd": ("bwd", 1.0, None),
    "bwd_drop": ("bwd", 0.9, None),
}
PARTS = {"fwd": ("o",), "bwd": ("dq", "dk", "dv")}
SEED = 0x1234_5678_9ABC


# --------------------------------------------------------------------------- cases
class Case:
    """One kernel call.  styles[h % len(styles)] picks how head h's inputs are drawn (see make_inputs)."""

    def __init__(self, name, NH, lens=None, L=None, mask=None, scale=None, styles=("random",), seed=0):
        self.name, self.NH, self.styles, self.seed = name, NH, styles, seed
        self.scale = 1.0 / math.sqrt(D) if scale is None else scale
        self.custom_scale = scale is not None
        if lens is not None:
            self.layout, self.lens = "packed", list(lens)
            self.B, self.L, self.T = len(lens), max(lens), sum(lens)
            self.cu = [0] + list(np.cumsum(lens))
            self.mask = None
        else:
            self.layout, self.mask = "padded", torch.as_tensor(mask, dtype=torch.int32)
            self.B, self.L = self.mask.shape
            self.T = self.B * self.L
            self.lens, self.cu = None, None

    def spans(self):
        """[(b, first row, length, additive key bias [length] float64)]"""
        out = []
        for b in range(self.B):
            if self.layout == "packed":
                n = self.lens[b]
                out.append((b, int(self.cu[b]), n, torch.zeros(n, dtype=torch.float64)))
            else:
                out.append((b, b * self.L, self.L, (1.0 - self.mask[b].double()) * MASK_ADD))
        return out

    def __repr__(self):
        return self.name


def _holes_mask(B, L, seed):
    """row 0 all valid, row 1 all masked, row 2 a valid prefix with holes, further rows ragged prefixes"""
    g = torch.Generator().manual_seed(seed)
    m = torch.zeros(B, L, dtype=torch.int32)
    for b in range(B):
        if b == 0:
            m[b] = 1
        elif b == 2:
            n = max(1, (3 * L) // 4)
            m[b, :n] = (torch.rand(n, generator=g) < 0.7).to(torch.int32)
            m[b, 0] = 1
        elif b > 2:
            m[b, :max(1, L // (b + 1))] = 1
    return m


def _ragged_mask(B, L):
    """row 0 all valid, the others valid prefixes of about 2/3, 1/3, ... of L"""
    m = torch.zeros(B, L, dtype=torch.int32)
    for b in range(B):
        m[b, :max(1, (L * (B - b)) // (B + 1)) if b else L] = 1
    return m


RAGGED = [1, 15, 16, 17, 31, 32, 33, 63, 0, 64, 65, 127, 128, 129, 191, 192, 255, 256, 0]
MIX = ("random", "peaked")

FWD_CASES = [   # every forward path (keys <= 256: the tcgen05 kernel's range)
    Case("packed_ragged_nh3", 3, lens=RAGGED, styles=("random", "peaked", "random"), seed=1),
    *[Case(f"padded_L{L}", 2, mask=_holes_mask(3, L, L), styles=MIX, seed=L) for L in (64, 128, 200, 256)],
    Case("packed_nh12", 12, lens=[5, 77, 130], styles=MIX, seed=2),
    Case("packed_nh1", 1, lens=[200, 3], seed=3),
    Case("packed_scale0.3", 2, lens=[40, 100], scale=0.3, styles=MIX, seed=4),
    Case("padded_scale0.2", 1, mask=_holes_mask(3, 96, 96), scale=0.2, styles=("peaked",), seed=5),
    Case("packed_sink", 2, lens=[2, 40, 130], styles=("sink",), seed=6),
]
FWD_LONG_CASES = [   # the mma.sync forward only (keys > 256)
    Case("packed_long", 2, lens=[257, 300, 384, 512, 768, 3], styles=MIX, seed=7),
    *[Case(f"padded_L{L}", 2 if B == 1 else 1, mask=_holes_mask(B, L, L), styles=MIX, seed=L)
      for L, B in ((257, 3), (300, 1), (384, 3), (512, 1), (768, 2))],
    Case("packed_long_sink", 1, lens=[700, 5], styles=("sink",), seed=8),
]
BWD_CASES = [
    *[Case(f"padded_L{L}", 2, mask=_ragged_mask(2, L), styles=MIX, seed=100 + L)
      for L in (1, 16, 17, 63, 64, 65, 128, 129, 200, 256, 300, 384)],
    Case("padded_holes_L96", 2, mask=_holes_mask(3, 96, 9), styles=MIX, seed=9),
    Case("packed_ragged_nh3", 3, lens=[1, 16, 17, 63, 0, 64, 65, 128, 129, 200, 256, 300, 384],
         styles=("random", "peaked", "random"), seed=10),
    Case("packed_mixed_nh1", 1, lens=[384, 7, 129, 2, 250, 0], seed=11),
    Case("packed_nh12", 12, lens=[150, 33, 260], styles=MIX, seed=12),
    Case("packed_scale0.3", 2, lens=[90, 17], scale=0.3, styles=MIX, seed=13),
    Case("packed_sink", 2, lens=[2, 40, 130, 300], styles=("sink",), seed=14),
]


def cases_for(path):
    if path == "fwd_tc":
        return FWD_CASES
    if path.startswith("fwd"):
        return FWD_CASES + FWD_LONG_CASES
    return BWD_CASES


def make_inputs(case):
    """-> (qkv bf16 [T, 3*NH*64], d_ctx bf16 [T, NH*64]) on the CPU.
    random: q, k, v ~ N(0, 1): scores ~ N(0, 1), flat rows (the bf16-rounding worst case of long sums).
    peaked: q_i = k_i: query i's argmax is key i (score ~ 8 against ~ N(0, 1)), so every key, the last one, key 64 and a
            key leaking in from the next rows move some output row by O(|v|); v scaled by 1/4 to keep |ctx| near the
            random heads'.
    sink:   key 0 of each sequence is zero with v_0 = e^10 u, query i >= 1 scores 10 on key i and query 0 scores 10 on key 1,
            so ctx_i ~ v_i + u with u weighted by e^(-10 * scale / scale0): the output moves by 20 % of u when scale does by 2 %."""
    NH, T = case.NH, case.T
    g = torch.Generator().manual_seed(1000 + case.seed)
    x = torch.randn(T, 3, NH, D, generator=g, dtype=torch.float64)
    dout = torch.randn(T, NH, D, generator=g, dtype=torch.float64)
    for h in range(NH):
        style = case.styles[h % len(case.styles)]
        if style == "peaked":
            x[:, 0, h] = x[:, 1, h] * (1.0 / (8.0 * case.scale))
            x[:, 2, h] *= 0.25
        elif style == "sink":
            gap = 10.0
            khat = x[:, 1, h] / x[:, 1, h].norm(dim=-1, keepdim=True)
            x[:, 1, h] = khat * 8.0
            x[:, 0, h] = khat * (gap / (8.0 * case.scale))
            for b, r0, n, _ in case.spans():
                if n < 2:
                    continue
                x[r0, 0, h] = khat[r0 + 1] * (gap / (8.0 * case.scale))
                x[r0, 1, h] = 0.0
                x[r0, 2, h] = x[r0, 2, h] * math.exp(gap)
    qkv = x.reshape(T, 3 * NH * D).to(torch.bfloat16)
    return qkv, dout.reshape(T, NH * D).to(torch.bfloat16)


# --------------------------------------------------------------------------- dropout
def keep_z(b, NH, Lq, Lk, keep, seed):
    """z(b, h, q, k) for h < NH, q < Lq, k < Lk as float64 [NH, Lq, Lk]: 1/keep (fp32, as the kernels compute it) or 0."""
    if keep >= 1.0:
        return torch.ones(NH, Lq, Lk, dtype=torch.float64)
    m32 = np.uint64(0xFFFFFFFF)
    lo, hi = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    bh = (np.uint64(b * NH) + np.arange(NH, dtype=np.uint64)).reshape(NH, 1, 1)
    sa = lo ^ ((bh * np.uint64(0x9E3779B1)) & m32)
    q = np.arange(Lq, dtype=np.uint64).reshape(1, Lq, 1)
    k = np.arange(Lk, dtype=np.uint64).reshape(1, 1, Lk)
    kept = hash3(sa, q, k ^ hi) < keep_threshold(keep)
    inv = float(np.float32(1.0) / np.float32(keep))
    return torch.from_numpy(kept.astype(np.float64) * inv)


# --------------------------------------------------------------------------- per-sequence operands (+ mutations)
FWD_MUTATIONS = ("drop_last_key", "drop_key64", "leak_next_row", "shift_row_base", "swap_v_heads", "scale_x1.02")
BWD_MUTATIONS = FWD_MUTATIONS + ("zero_dk_tile", "z_transposed", "z_in_dv_only")
DROP_ONLY = ("z_transposed", "z_in_dv_only")


def mutations_for(path):
    muts = FWD_MUTATIONS if path.startswith("fwd") else BWD_MUTATIONS
    return [m for m in muts if PATHS[path][1] < 1.0 or m not in DROP_ONLY]


def _split(qkv, NH):
    x = qkv.double().reshape(-1, 3, NH, D)
    return x[:, 0], x[:, 1], x[:, 2]


def _operands(case, Q, K, V, span, keep, seed, mut, shift_b):
    """q [NH, n, D], k / v [NH, nk, D], key bias [nk], z [NH, n, nk], scale for one sequence, with `mut` applied."""
    b, r0, n, bias = span
    T = Q.shape[0]
    scale = case.scale * (1.02 if mut == "scale_x1.02" else 1.0)
    qrows = krows = torch.arange(r0, r0 + n)
    bias = bias.clone()
    if mut == "shift_row_base" and b == shift_b:
        qrows = krows = qrows + 1
    if mut == "drop_last_key" and n >= 2:
        bias[n - 1] = -math.inf
    if mut == "drop_key64" and n > 64:
        bias[64] = -math.inf
    if mut == "leak_next_row" and r0 + n < T:
        krows = torch.arange(r0, r0 + n + 1)
        bias = torch.cat([bias, torch.zeros(1, dtype=torch.float64)])
    q, k, v = Q[qrows].transpose(0, 1), K[krows].transpose(0, 1), V[krows].transpose(0, 1)
    if mut == "swap_v_heads" and case.NH >= 2:
        v = v[[1, 0] + list(range(2, case.NH))]
    z = keep_z(b, case.NH, n, len(krows), keep, seed)
    return q, k, v, bias, z, scale


def _shift_target(case):
    """the packed sequence whose row_base the shift mutation moves: the second one that has rows and room after it"""
    if case.layout != "packed":
        return None
    for b, r0, n, _ in case.spans():
        if b >= 1 and n >= 1 and r0 + n + 1 <= case.T:
            return b
    return None


def applies(case, mut):
    if mut == "shift_row_base":
        return _shift_target(case) is not None
    if mut == "swap_v_heads":
        return case.NH >= 2
    return True


# --------------------------------------------------------------------------- reference forward / backward
def _probs(q, k, bias, scale):
    return torch.softmax(scale * (q @ k.transpose(-1, -2)) + bias, dim=-1)


def forward(case, qkv, keep=1.0, seed=SEED, mut=None):
    """ctx as float64 [T, NH, D]"""
    Q, K, V = _split(qkv, case.NH)
    out = torch.zeros(case.T, case.NH, D, dtype=torch.float64)
    sb = _shift_target(case)
    for span in case.spans():
        if span[2] == 0:
            continue
        q, k, v, bias, z, scale = _operands(case, Q, K, V, span, keep, seed, mut, sb)
        out[span[1]:span[1] + span[2]] = ((_probs(q, k, bias, scale) * z) @ v).transpose(0, 1)
    return out


def backward(case, qkv, dout, keep=1.0, seed=SEED):
    """torch autograd of forward(): (dQ, dK, dV) as float64 [T, NH, D] each, plus ctx"""
    Q, K, V = (t.clone().requires_grad_(True) for t in _split(qkv, case.NH))
    out = torch.zeros(case.T, case.NH, D, dtype=torch.float64)
    for span in case.spans():
        if span[2] == 0:
            continue
        q, k, v, bias, z, scale = _operands(case, Q, K, V, span, keep, seed, None, None)
        out[span[1]:span[1] + span[2]] = ((_probs(q, k, bias, scale) * z) @ v).transpose(0, 1)
    grads = torch.autograd.grad(out, (Q, K, V), dout.double().reshape(case.T, case.NH, D), allow_unused=True)
    return tuple(torch.zeros_like(Q) if g_ is None else g_.detach() for g_ in grads) + (out.detach(),)


def backward_closed(case, qkv, dout, keep=1.0, seed=SEED, mut=None, ctx=None):
    """DESIGN.md 3.5 in float64: dS = P o (z o dP - D), dV = (P o z)^T dO, D = rowsum(dO o O), dQ = scale dS K,
    dK = scale dS^T Q.  O is `ctx` ([T, NH*D], e.g. the bf16 context the kernel is given) or the exact forward.
    Gradients reaching rows outside the sequence (leak mutation) are dropped."""
    Q, K, V = _split(qkv, case.NH)
    dO_all = dout.double().reshape(case.T, case.NH, D)
    O_all = forward(case, qkv, keep, seed) if ctx is None else ctx.double().reshape(case.T, case.NH, D)
    dq, dk, dv = (torch.zeros(case.T, case.NH, D, dtype=torch.float64) for _ in range(3))
    sb = _shift_target(case)
    for span in case.spans():
        b, r0, n, _ = span
        if n == 0:
            continue
        q, k, v, bias, z, scale = _operands(case, Q, K, V, span, keep, seed, mut, sb)
        zs = z.transpose(-1, -2)[:, :, :n] if mut == "z_transposed" and z.shape[-1] == n else z
        zv = zs
        if mut == "z_in_dv_only":
            zs = torch.ones_like(z)
        rows = slice(r0, r0 + n)
        dO, O = dO_all[rows].transpose(0, 1), O_all[rows].transpose(0, 1)
        P = _probs(q, k, bias, scale)
        Dr = (dO * O).sum(-1, keepdim=True)
        dS = P * (zs * (dO @ v.transpose(-1, -2)) - Dr)
        dq[rows] = (scale * dS @ k).transpose(0, 1)
        dk_s = (scale * dS.transpose(-1, -2) @ q)[:, :n]
        dv_s = ((P * zv).transpose(-1, -2) @ dO)[:, :n]
        if mut == "zero_dk_tile":
            t = (n - 1) // 16
            dk_s[:, 16 * t:16 * t + 16] = 0.0
        dk[rows] = dk_s.transpose(0, 1)
        dv[rows] = dv_s.transpose(0, 1)
    return dq, dk, dv


# --------------------------------------------------------------------------- kernel emulations
def _bf16(x):
    return x.to(torch.bfloat16).double()


def _f32(x):
    return x.float().double()


def emulate_fwd_tc(case, qkv):
    """attention_tc.cu: x = scores * scale * log2e + madd * log2e in fp32, unnormalised P = 2^(x - rowmax) rounded to bf16
    for P V, row sum of the unrounded p, ctx = bf16(O / sum)."""
    Q, K, V = _split(qkv, case.NH)
    out = torch.zeros(case.T, case.NH, D, dtype=torch.float64)
    for b, r0, n, bias in case.spans():
        if n == 0:
            continue
        q, k, v = (t[r0:r0 + n].transpose(0, 1) for t in (Q, K, V))
        x = _f32(_f32(q @ k.transpose(-1, -2)) * _f32(torch.tensor(case.scale * LOG2E)) + _f32(bias * LOG2E))
        p = torch.exp2(x - x.amax(-1, keepdim=True))
        out[r0:r0 + n] = _bf16((_bf16(p) @ v) / p.sum(-1, keepdim=True)).transpose(0, 1)
    return out


def emulate_fwd_mma(case, qkv, keep=1.0, seed=SEED):
    """attention.cu in its flash order: per 64-key block, P = exp(s - running max) (times z) rounded to bf16 for P V; the row
    sum of the unrounded, undropped p; ctx = bf16(O / sum)."""
    Q, K, V = _split(qkv, case.NH)
    out = torch.zeros(case.T, case.NH, D, dtype=torch.float64)
    for b, r0, n, bias in case.spans():
        if n == 0:
            continue
        nb = (n + 63) // 64
        q, k, v = (t[r0:r0 + n].transpose(0, 1) for t in (Q, K, V))
        s = _f32(_f32(q @ k.transpose(-1, -2)) * case.scale + bias)
        s = torch.nn.functional.pad(s, (0, nb * 64 - n), value=-1e30).reshape(case.NH, n, nb, 64)
        m = torch.cummax(s.amax(-1), dim=-1).values                  # running max after each block
        p = torch.exp(s - m[..., None])
        w = torch.exp(m - m[..., -1:])                               # rescale of each block's partial sums to the final max
        z = torch.nn.functional.pad(keep_z(b, case.NH, n, n, keep, seed), (0, nb * 64 - n)).reshape(case.NH, n, nb, 64)
        vb = torch.nn.functional.pad(v, (0, 0, 0, nb * 64 - n)).reshape(case.NH, nb, 64, D)
        o = (torch.einsum("hqjk,hjkd->hqjd", _bf16(p * z), vb) * w[..., None]).sum(-2)
        l = (p.sum(-1) * w).sum(-1, keepdim=True)
        out[r0:r0 + n] = _bf16(o / l).transpose(0, 1)
    return out


def emulate_bwd(case, qkv, dout, ctx, keep=1.0, seed=SEED):
    """attention_bwd.cu: fp32 scores, P = exp(s - max) / sum, D = rowsum(dO o ctx) from the bf16 ctx it is given,
    dS = P o (z o dP - D) and P o z rounded to bf16 where mma_p_b packs them, dQ / dK / dV rounded to bf16."""
    Q, K, V = _split(qkv, case.NH)
    dO_all = dout.double().reshape(case.T, case.NH, D)
    O_all = ctx.double().reshape(case.T, case.NH, D)
    dq, dk, dv = (torch.zeros(case.T, case.NH, D, dtype=torch.float64) for _ in range(3))
    for b, r0, n, bias in case.spans():
        if n == 0:
            continue
        q, k, v, dO, O = (t[r0:r0 + n].transpose(0, 1) for t in (Q, K, V, dO_all, O_all))
        s = _f32(_f32(q @ k.transpose(-1, -2)) * case.scale + bias)
        p = torch.exp(s - s.amax(-1, keepdim=True))
        p = p / p.sum(-1, keepdim=True)
        z = keep_z(b, case.NH, n, n, keep, seed)
        dS = _bf16(p * (z * (dO @ v.transpose(-1, -2)) - (dO * O).sum(-1, keepdim=True)))
        dq[r0:r0 + n] = _bf16(case.scale * dS @ k).transpose(0, 1)
        dk[r0:r0 + n] = _bf16(case.scale * dS.transpose(-1, -2) @ q).transpose(0, 1)
        dv[r0:r0 + n] = _bf16(_bf16(p * z).transpose(-1, -2) @ dO).transpose(0, 1)
    return dq, dk, dv


# --------------------------------------------------------------------------- bound
def block_max(case, X64):
    """per (sequence, head) block: max |X64| [nblk], in the order of block_stats"""
    return torch.cat([X64[r0:r0 + n].abs().amax(dim=(0, 2)) for b, r0, n, _ in case.spans() if n > 0])


def floors(case, ref_parts):
    """{part: 2^-9 max|X64| per (sequence, head) block [nblk]}; a block whose part is identically zero (dQ and dK of a
    one-key sequence) takes the max over all parts of that block instead"""
    mx = {part: block_max(case, x) for part, x in ref_parts.items()}
    whole = torch.stack(list(mx.values())).amax(0)
    return {part: FLOOR * torch.where(m > 0, m, whole) for part, m in mx.items()}


def block_stats(case, X, X64):
    """per (sequence, head) block: (err [nblk], rms [nblk], labels)"""
    errs, rmss, labels = [], [], []
    for b, r0, n, _ in case.spans():
        if n == 0:
            continue
        d = torch.nan_to_num((X[r0:r0 + n] - X64[r0:r0 + n]).abs(), nan=math.inf)
        errs.append(d.amax(dim=(0, 2)))
        rmss.append(X64[r0:r0 + n].pow(2).mean(dim=(0, 2)).sqrt())
        labels += [(b, n, h) for h in range(case.NH)]
    return torch.cat(errs), torch.cat(rmss), labels


def worst_ratio(case, outs, refs, path):
    """max over parts and blocks of err / bound with tau = TAU[path, part]; -> (ratio, (part, (b, len, head)))"""
    fl = floors(case, refs)
    worst, where = 0.0, None
    for part in refs:
        err, rms, labels = block_stats(case, outs[part], refs[part])
        bound = TAU[(path, part)] * rms + fl[part]
        # a block that is exactly zero in every part (one key, dropped) has bound 0: only an exact 0 passes
        ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
        i = int(torch.argmax(ratio))
        if float(ratio[i]) > worst or where is None:
            worst, where = float(ratio[i]), (part, labels[i])
    return worst, where


def needed_tau(case, outs, refs):
    """{part: smallest tau for which outs pass the bound}"""
    fl = floors(case, refs)
    need = {}
    for part in refs:
        err, rms, _ = block_stats(case, outs[part], refs[part])
        excess = (err - fl[part]).clamp(min=0.0)
        need[part] = float(torch.where(excess > 0, excess / rms, torch.zeros_like(rms)).max())
    return need


# --------------------------------------------------------------------------- per-path drivers
def ctx_for_bwd(case, qkv, keep):
    """the bf16 context the backward tests hand to the kernel: the exact forward, rounded"""
    return forward(case, qkv, keep).reshape(case.T, case.NH * D).to(torch.bfloat16)


def reference(case, path, qkv, dout):
    """{part: X64} of the path.  The backward kernel is handed the context and takes D = rowsum(dO o ctx) from it, so its
    reference is the closed form with that same bf16 ctx (the autograd gradient of the exact forward differs from it by
    the rounding of ctx alone, up to ~20 % of dQ's RMS on a saturated head)."""
    direction, keep, _ = PATHS[path]
    if direction == "fwd":
        return {"o": forward(case, qkv, keep)}
    dq, dk, dv = backward_closed(case, qkv, dout, keep, ctx=ctx_for_bwd(case, qkv, keep))
    return {"dq": dq, "dk": dk, "dv": dv}


def emulation(case, path, qkv, dout):
    direction, keep, variant = PATHS[path]
    if path == "fwd_tc":
        return {"o": emulate_fwd_tc(case, qkv)}
    if direction == "fwd":
        return {"o": emulate_fwd_mma(case, qkv, keep)}
    dq, dk, dv = emulate_bwd(case, qkv, dout, ctx_for_bwd(case, qkv, keep), keep)
    return {"dq": dq, "dk": dk, "dv": dv}


def mutated(case, path, qkv, dout, mut):
    direction, keep, _ = PATHS[path]
    if direction == "fwd":
        return {"o": forward(case, qkv, keep, mut=mut)}
    dq, dk, dv = backward_closed(case, qkv, dout, keep, mut=mut, ctx=ctx_for_bwd(case, qkv, keep))
    return {"dq": dq, "dk": dk, "dv": dv}
