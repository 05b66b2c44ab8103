"""Every compiled attention kernel element by element against a float64 reference.

Kernels and the entries that force them:
  attn_tc.cu      16 kernels: exp2 masks 0x00, 0x88, 0xA8, 0xAA (bit p % 8 set: pair p of a score row takes the FMA-pipe
                  polynomial instead of the MUFU), times plain (128-key blocks) and pair (64-key blocks, two value
                  tensors), times bf16 and fp16.  ops.attention / ops.attention_pair with variant 1, 2 -> 0x00,
                  3 -> 0x88, 0, 4 -> 0xA8, 5 -> 0xAA (the aliases are checked to give the same bits).
  attn_wide.cu    head_dim 512, bf16 and fp16 (ops.attention_d512).
  attn_d80.cu     head_dim 80, bf16 and fp16 (ops.attention_d80).
  attn_temporal   TP = 16 / 32 x exact / masked, bf16 (ops.temporal_attention, ops.temporal_attention_frames: T = 16,
                  32 and T in 1..15, 17..31).
  inject.cu       ops.attention_inject_: spatial with and without the shared softmax, and temporal.

The reference, per (batch, head) and in float64 from the same 16-bit inputs: s = scale q k^T, pi = softmax(s),
ref = pi v, A = pi |v|.  Every output element must satisfy

    |out - ref| <= u |ref| + (u + E + 2^-16 + 2 delta_i) A + sigma sum_k |v_kc| / sum_k exp(s_ik - max_k s_ik)

  u |ref|     the one rounding of the output (u = 2^-8 bf16, 2^-11 fp16; the fp32 1/l and the product by it are two
              more roundings of 2^-24, inside the 2^-16 A below since A >= |ref|).
  u A         P is rounded to the storage type before P V: each p_k moves by at most u p_k, so the output by
              u sum p_k |v_k| / l = u A.
  E A         the exp2 error e enters p (numerator) and the row sum l separately, because l is summed from the
              unrounded p: E = 2 e.  ex2.approx.ftz.f32 and exp2f (temporal kernel): e = 2^-22.  The degree-3
              polynomial ptx::ex2_poly2: e = its largest relative error on [0, 1) (poly_error(), computed below from
              the coefficients in float64) plus 3 fp32 roundings of the Horner steps; the integer part is exact.
  2^-16 A     fp32 accumulation of P V in the tensor cores (the allowance of the GEMM matrix, relative to the same
              sum of absolute values).
  2 delta_i A a score error of at most delta on every key moves each weight pi_k by a factor within e^(+-2 delta).
              delta_i = 2^-16 scale max_k(|q_i| |k_k|^T) for the fp32 accumulation of Q K^T, plus 5 2^-24 max_k |s_ik|
              for the fp32 argument of exp2: x = fma(s, sl2, -m sl2) rounds -m sl2 and x (|x| <= 2 max |s| sl2), and
              sl2 = scale log2(e) is itself rounded (an error of 2^-24 |s - m| sl2 <= 2^-23 max |s| sl2).
  sigma term  P underflow: a p below the smallest normal of P's type keeps only an absolute precision sigma
              (fp16: half the subnormal spacing, 2^-25; bf16, and the flush to zero of ex2.approx.ftz: 2^-126), so
              the output moves by sigma sum_k |v_kc| / l.  The kernels' lagging maximum m_used <= max s keeps the
              largest p >= 1, so l >= sum_k exp(s_ik - max s_ik).
The lazy rescale (threshold 8 in log2) only lets p grow up to 2^8 between rescales, so it needs no term of its own; the
rescale factor multiplies O and l alike.  test_emulation_inside_the_bound and test_mutants_break_the_bound show, on the
CPU, that a float32 emulation of the head_dim-64 kernel passes this bound on every input kind while a dropped key,
unmasked padding keys, a skipped rescale and a V row one key off at a block edge fail it.

Inputs (every shape runs each kind):
  random      Gaussian q, k, v; logits span a few units.
  uniform     q = 0: the reference is the mean of v over the valid keys.  v has mean 1, so padding keys (TMA zero
              fill) in the row sum, or a valid key masked off, move the output by a visible share when few keys are
              valid.
  retrieval   keys of random +-1 entries (one norm), q_i = 4 k_sigma(i): >= 0.99 of the weight on key sigma(i)
              (asserted in float64), so out_i ~ v_sigma(i).  Across the (batch, head, query) rows of a case sigma covers
              key 0, the last key, both sides of every 64-key edge and, given enough rows, every key: a dropped,
              duplicated or shifted K or V row fails by order 1.  The logits are large, so the rescale runs too.
  ramp        the logits step up by 1.25 x 8 log2 units at a third, at two thirds and at the last key block: the
              running maximum jumps past the rescale threshold, once in the last block.
  ramp_under  the same steps at 0.9 x 8: no rescale at the first step, so p reaches about 2^7.

Harness: q, k, v are views into NaN-guarded allocations (with the strides of fused QKV column slices in the fused
layout) and stay bit-identical; the output is a NaN-guarded view that only the kernel's rows and columns may change
(the pair case with pair_batches > B also leaves the output batches in between); two calls give the same bits; one
batch run alone gives the same bits as inside the full call; pair: v[b] == v[b + pair_batches] gives two identical
outputs."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.test_gemm_matrix_gpu import DTYPES, UNIT, Guarded, run_twice

HD = 64
ACC = 2.0 ** -16                                 # fp32 accumulation allowance (Q K^T and P V)
SCORE_FP32 = 5 * 2.0 ** -24                      # fp32 argument of exp2, relative to max |s|
EX2_ERR = 2.0 ** -22                             # ex2.approx.ftz.f32, exp2f
SIGMA = {torch.bfloat16: 2.0 ** -126, torch.float16: 2.0 ** -25}
POLY = (0.077119089663028717041015625, 0.227564394474029541015625, 0.695146143436431884765625, 1.0)   # ptx.cuh
RESCALE_LOG2 = 8.0
VARIANT_MASK = {0: 0xA8, 1: 0x00, 2: 0x00, 3: 0x88, 4: 0xA8, 5: 0xAA}
MASK_VARIANT = {0x00: 1, 0x88: 3, 0xA8: 0, 0xAA: 5}
KINDS = ("random", "uniform", "retrieval", "ramp", "ramp_under")
REDUCED_KINDS = ("retrieval", "uniform", "ramp")


def poly_error():
    """Largest relative error of ptx::ex2_poly2 on the fraction [0, 1): the polynomial's own error in float64 over a
    2^22-point grid, plus three fp32 roundings of its Horner steps (results in [1, 2))."""
    f = torch.arange(2 ** 22, dtype=torch.float64) / 2 ** 22
    c = [float(torch.tensor(x, dtype=torch.float32)) for x in POLY]
    p = ((c[0] * f + c[1]) * f + c[2]) * f + c[3]
    return float((p / torch.exp2(f) - 1).abs().max()) + 3 * 2.0 ** -24


def exp2_bound(mask):
    """E: twice the exp2 error of a kernel whose pairs selected by `mask` take the polynomial."""
    return 2 * max(EX2_ERR, poly_error() if mask else 0.0)


def f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


# ------------------------------------------------------------------ inputs
def retrieval_keys(rows, nk, gen):
    """The chosen key of each of `rows` query rows: first key 0, the last key and both sides of every 64-key edge, then
    the other keys in random order, repeated."""
    first = [0, nk - 1] + [i for e in range(64, nk, 64) for i in (e - 1, e)]
    first = list(dict.fromkeys(first))
    rest = torch.tensor(sorted(set(range(nk)) - set(first)), dtype=torch.long)
    perm = torch.cat([torch.tensor(first, dtype=torch.long), rest[torch.randperm(len(rest), generator=gen)]])
    return perm[torch.arange(rows) % nk]


def ramp_levels(nk, step):
    """Logit level of each key: `step` more at a third, at two thirds and at the last 128-key block."""
    nb = -(-nk // 128)
    jumps = sorted({nb // 3, 2 * nb // 3, nb - 1} - {0})
    blk = torch.arange(nk) // 128
    return step * sum((blk >= j).double() for j in jumps) if jumps else torch.zeros(nk, dtype=torch.float64)


def make_inputs(kind, B, H, Nq, Nk, D, Bv, dev, seed):
    """float32 q [B, Nq, H*D], k [B, Nk, H*D], v [Bv, Nk, H*D] of one input kind (rounded when stored)."""
    gen = torch.Generator().manual_seed(seed)
    g = lambda *s: torch.randn(*s, generator=gen)
    scale = D ** -0.5
    if kind == "random":
        q, k, v = 2 * g(B, H, Nq, D), g(B, H, Nk, D), g(Bv, H, Nk, D)
    elif kind == "uniform":
        q, k, v = torch.zeros(B, H, Nq, D), g(B, H, Nk, D), 1 + 0.25 * g(Bv, H, Nk, D)
    elif kind == "retrieval":
        k = torch.randint(0, 2, (B, H, Nk, D), generator=gen).float() * 2 - 1
        sel = retrieval_keys(B * H * Nq, Nk, gen).view(B, H, Nq, 1).expand(-1, -1, -1, D)
        q, v = 4 * torch.gather(k, 2, sel), g(Bv, H, Nk, D)
    else:
        step = (1.25 if kind == "ramp" else 0.9) * RESCALE_LOG2 * math.log(2)
        q, k, v = 0.5 * g(B, H, Nq, D), 0.25 * g(B, H, Nk, D), g(Bv, H, Nk, D)
        q[..., 0] = 1
        k[..., 0] = ramp_levels(Nk, step).float() / scale
    to = lambda t: t.permute(0, 2, 1, 3).reshape(t.shape[0], t.shape[2], H * D).to(dev)
    return to(q), to(k), to(v)


def groups(t, H, D):
    """[B, N, H*D] -> [B*H, N, D]: one (batch, head) problem per group."""
    B, N = t.shape[0], t.shape[1]
    return t.reshape(B, N, H, D).permute(0, 2, 1, 3).reshape(B * H, N, D)


# ------------------------------------------------------------------ reference and bound
def reference(q, k, v, scale, dtype, E):
    """q [G, Nq, D], k [G, Nk, D], v [G, Nk, Dv] (16-bit, any device) -> float64 ref, bound and the largest softmax
    weight of every row, in chunks of query rows."""
    G, Nq, _ = q.shape
    Nk = k.shape[1]
    qd, kd, vd = q.double(), k.double(), v.double()
    ka, va = kd.abs().transpose(1, 2), vd.abs()
    v1 = va.sum(1, keepdim=True)
    u = UNIT[dtype]
    ref = torch.empty(G, Nq, vd.shape[2], dtype=torch.float64, device=q.device)
    bound, top = torch.empty_like(ref), torch.empty(G, Nq, dtype=torch.float64, device=q.device)
    step = max(1, 2 ** 26 // (G * Nk))
    for i in range(0, Nq, step):
        qc = qd[:, i:i + step]
        s = scale * (qc @ kd.transpose(1, 2))
        e = torch.exp(s - s.amax(-1, keepdim=True))
        den = e.sum(-1, keepdim=True)
        pi = e / den
        r, A = pi @ vd, pi @ va
        delta = ACC * scale * (qc.abs() @ ka).amax(-1, keepdim=True) + SCORE_FP32 * s.abs().amax(-1, keepdim=True)
        ref[:, i:i + step] = r
        bound[:, i:i + step] = u * r.abs() + (u + E + ACC + 2 * delta) * A + SIGMA[dtype] * v1 / den
        top[:, i:i + step] = pi.amax(-1)
    return ref, bound, top


def max_ratio(out, ref, bound):
    return float(((out.double() - ref).abs() / bound.clamp_min(torch.finfo(torch.float64).tiny)).max())


def check_attention(desc, out, ref, bound, H, nk_blocks, batches=None):
    """out, ref, bound: [G, Nq, Dv] with group g = (batch, head) = divmod(g, H) (batch relabelled through `batches`).
    Returns the largest err / bound."""
    out = out.double()
    label = lambda g: f"(batch, head) = ({g // H if batches is None else batches[g // H]}, {g % H})"
    bad = ~torch.isfinite(out)
    if bool(bad.any()):
        g, i, c = (int(x) for x in bad.nonzero()[0])
        raise AssertionError(f"{desc}: {int(bad.sum())} outputs are not finite (a read beside an operand or an "
                             f"unwritten row), the first at {label(g)} query row {i} column {c}")
    ratio = (out - ref).abs() / bound.clamp_min(torch.finfo(torch.float64).tiny)
    worst = int(ratio.argmax())
    r = float(ratio.reshape(-1)[worst])
    if r > 1.0:
        g, rem = divmod(worst, ratio.shape[1] * ratio.shape[2])
        i, c = divmod(rem, ratio.shape[2])
        raise AssertionError(
            f"{desc}: worst element at {label(g)} query row {i} column {c} (query tile {i // 128}, {nk_blocks} key "
            f"blocks): out {float(out[g, i, c]):.6g} ref {float(ref[g, i, c]):.6g} bound {float(bound[g, i, c]):.3g}, "
            f"err / bound = {r:.3g}")
    return r


def verify(desc, kind, out_g, q_g, k_g, v_g, scale, dtype, E, H, nk_blocks, batches=None):
    ref, bound, top = reference(q_g, k_g, v_g, f32(scale), dtype, E)
    if kind == "retrieval":
        assert float(top.min()) >= 0.99, f"{desc}: retrieval input puts only {float(top.min()):.3f} on its key"
    r = check_attention(desc, out_g, ref, bound, H, nk_blocks, batches)
    print(f"[attention matrix] {desc}: max err/bound {r:.4f}")
    return r


def same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16))


# ------------------------------------------------------------------ the CPU emulation of attn_tc.cu and its mutants
def fma32(a, b, c):
    """fp32 fma: the float64 product of two fp32 values is exact, one rounding to fp32."""
    return (a.double() * b.double() + c.double()).float()


def ex2_poly32(x):
    """ptx::ex2_poly2 in fp32: clamp at -127, floor, Horner on the fraction, the integer part into the exponent."""
    xc = x.clamp_min(-127.0)
    fl = torch.floor(xc)
    xf = xc - fl
    c = [torch.tensor(v, dtype=torch.float32) for v in POLY]
    p = fma32(fma32(fma32(c[0], xf, c[1]), xf, c[2]), xf, c[3])
    return torch.ldexp(p, fl)


def emulate_attn_tc(q, k, v, scale, dtype, mask, mutant=None):
    """The plain head_dim-64 kernel's arithmetic in fp32 on [G, N, 64] groups: 128-key blocks, TMA zero fill and -inf
    tail scores, the lagging maximum with a log2 threshold of 8, exp2 on the MUFU or (pairs selected by `mask`) the
    polynomial, l summed from the unrounded p, P rounded to the storage type, the output rounded once.
    Mutants: drop_last (the last key masked off), no_tail_mask (padding keys in the row sum), no_rescale (the maximum
    moves but O and l are not rescaled), v_edge (key 128 multiplies the V row of key 129)."""
    BN = 128
    G, Nq, _ = q.shape
    Nk = k.shape[1]
    nb = -(-Nk // BN)
    kp = F.pad(k.double(), (0, 0, 0, nb * BN - Nk))
    vp = F.pad(v.float(), (0, 0, 0, nb * BN - Nk))
    if mutant == "v_edge":
        vp[:, 128] = vp[:, 129]
    sl2 = torch.tensor(f32(scale), dtype=torch.float32) * torch.tensor(1.4426950408889634, dtype=torch.float32)
    s_all = (q.double() @ kp.transpose(1, 2)).float()
    emu = torch.tensor([(mask >> ((c // 2) % 8)) & 1 for c in range(BN)], dtype=torch.bool)
    m_used = l = O = None
    for j in range(nb):
        s = s_all[..., j * BN:(j + 1) * BN].clone()
        valid = min(BN, Nk - j * BN) - (mutant == "drop_last" and j == nb - 1)
        if mutant != "no_tail_mask":
            s[..., valid:] = -math.inf
        mx = s.amax(-1)
        if j == 0:
            m_used, l, O = mx, torch.zeros(G, Nq), torch.zeros(G, Nq, v.shape[2])
        else:
            m_new = torch.maximum(m_used, mx)
            need = (m_new - m_used) * sl2 > RESCALE_LOG2
            if mutant != "no_rescale":
                f = torch.where(need, torch.exp2((m_used - m_new) * sl2), torch.ones(()))
                l, O = l * f, O * f[..., None]
            m_used = torch.where(need, m_new, m_used)
        x = fma32(s, sl2, (-m_used * sl2)[..., None])
        p = torch.where(emu, ex2_poly32(x), torch.exp2(x))
        l = l + p.sum(-1)
        O = O + (p.to(dtype).double() @ vp[:, j * BN:(j + 1) * BN].double()).float()
    return (O * (1.0 / l)[..., None]).to(dtype)


EMU_SHAPE = (1, 2, 160, 300)     # B, H, Nq, Nk: three key blocks, a ragged tail, 320 query rows cover every key


def emulation_case(kind, dtype, mask, mutant=None):
    B, H, Nq, Nk = EMU_SHAPE
    q, k, v = (t.to(dtype) for t in make_inputs(kind, B, H, Nq, Nk, HD, B, "cpu", seed=11))
    qg, kg, vg = groups(q, H, HD), groups(k, H, HD), groups(v, H, HD)
    out = emulate_attn_tc(qg, kg, vg, HD ** -0.5, dtype, mask, mutant)
    ref, bound, top = reference(qg, kg, vg, f32(HD ** -0.5), dtype, exp2_bound(mask))
    if kind == "retrieval":
        assert float(top.min()) >= 0.99
    return max_ratio(out, ref, bound)


@pytest.mark.parametrize("mask", [0x00, 0xA8])
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("kind", KINDS)
def test_emulation_inside_the_bound(kind, dt, mask):
    r = emulation_case(kind, DTYPES[dt], mask)
    print(f"emulation {kind} {dt} mask {mask:#04x}: max err/bound {r:.4f}")
    assert r <= 1.0


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("mutant,kind", [("drop_last", "retrieval"), ("no_tail_mask", "uniform"),
                                         ("no_rescale", "ramp"), ("v_edge", "retrieval")])
def test_mutants_break_the_bound(mutant, kind, dt):
    r = emulation_case(kind, DTYPES[dt], 0xA8, mutant)
    print(f"mutant {mutant} on {kind} {dt}: max err/bound {r:.1f}")
    assert r > 4.0, f"the bound does not see the {mutant} mutant (max err/bound {r:.3f})"


def test_poly_error_is_the_documented_one():
    e = poly_error()
    assert 8e-5 < e < 9.5e-5, e


# ------------------------------------------------------------------ head_dim 64: ops.attention and ops.attention_pair
# (B, H, Nq, Nk): every Nk of the list (ring of 3 stages: 384 fills it, 896 wraps it twice) and every Nq, H
PLAIN_SHAPES = [(2, 2, 129, 1), (1, 5, 127, 63), (2, 1, 1, 64), (1, 2, 129, 65), (2, 10, 127, 77), (1, 20, 129, 127),
                (3, 1, 1, 128), (1, 2, 880, 129), (2, 5, 880, 145), (1, 1, 4096, 384), (1, 2, 127, 385),
                (1, 5, 129, 896), (1, 2, 4096, 4096), (16, 5, 4096, 4096)]
# (B, H, Nq, Nk, pair_batches): pair_batches == B (the product's call) and > B
PAIR_SHAPES = [(2, 2, 129, 1, 2), (1, 5, 127, 63, 3), (2, 1, 1, 64, 2), (3, 2, 129, 65, 4), (2, 10, 127, 192, 2),
               (1, 2, 880, 193, 1), (2, 5, 129, 448, 3), (1, 2, 4096, 4096, 1), (2, 1, 880, 4096, 3)]
REDUCED_SHAPE = (2, 2, 129, 385)       # other masks: ragged query tile, four 128-key blocks (seven 64-key), ragged
LAYOUTS = ("separate", "fused")


def shape_id(s):
    return "x".join(map(str, s))


def tc_cases():
    """(mode, mask, dt, shape, layout, kind): the default mask on every shape, the other masks on the reduced set."""
    cases = []
    for mode, shapes in (("plain", PLAIN_SHAPES), ("pair", PAIR_SHAPES)):
        for dt in DTYPES:
            for shape in shapes:
                cases += [(mode, 0xA8, dt, shape, lay, kind) for lay in LAYOUTS for kind in KINDS]
            for mask in (0x00, 0x88, 0xAA):
                shape = REDUCED_SHAPE if mode == "plain" else REDUCED_SHAPE + (REDUCED_SHAPE[0],)
                cases += [(mode, mask, dt, shape, "fused", kind) for kind in REDUCED_KINDS]
    return cases


TC_CASES = tc_cases()


def tc_id(c):
    mode, mask, dt, shape, layout, kind = c
    return f"{mode}-{mask:#04x}-{dt}-{shape_id(shape)}-{layout}-{kind}"


def qkv_operands(q, k, v, dtype, dev, layout):
    """Guarded q, k, v: contiguous, or with the row stride of a fused [*, N, 3C] QKV output (NaN between the rows)."""
    ld = 3 * q.shape[-1] if layout == "fused" else None
    return tuple(Guarded(tuple(t.shape), dtype, dev, ld=ld, fill=t) for t in (q, k, v))


def out_maker(shape, dtype, dev, layout):
    return lambda: Guarded(shape, dtype, dev, ld=shape[-1] + 64 if layout == "fused" else None)


@pytest.mark.gpu
@pytest.mark.parametrize("case", TC_CASES, ids=tc_id)
def test_attention_tc_vs_float64(cuda_device, case):
    from mvoc_b200 import ops

    mode, mask, dt, shape, layout, kind = case
    dtype, dev, variant = DTYPES[dt], cuda_device, MASK_VARIANT[mask]
    pair = mode == "pair"
    B, H, Nq, Nk = shape[:4]
    pb = shape[4] if pair else 0
    C, Bv, scale = H * HD, B + pb, HD ** -0.5
    entry = "attention_pair" if pair else "attention"
    desc = (f"ops.{entry} {dt} mask {mask:#04x} {'pair, 64-key' if pair else 'plain, 128-key'} blocks, "
            f"B={B} H={H} Nq={Nq} Nk={Nk}{f' pair_batches={pb}' if pair else ''} {layout} {kind}")
    q, k, v = qkv_operands(*make_inputs(kind, B, H, Nq, Nk, HD, Bv, "cpu", seed=sum(shape) + mask), dtype, dev, layout)
    make_out = out_maker((Bv if pair else B, Nq, C), dtype, dev, layout)
    if pair:
        launch = lambda o, qq=q.t, kk=k.t, vv=v.t, p=pb: ops.attention_pair(qq, kk, vv, H, p, scale, o, variant)
    else:
        launch = lambda o, qq=q.t, kk=k.t, vv=v.t: ops.attention(qq, kk, vv, H, scale, o, variant)
    out = run_twice(desc, launch, make_out, {"q": q, "k": k, "v": v})
    if pair and pb > B:
        assert torch.isnan(out[B:pb]).all(), f"{desc}: output batches [B, pair_batches) were written"
    qg, kg = groups(q.t, H, HD), groups(k.t, H, HD)
    if pair:
        out_g = torch.cat([groups(out[:B], H, HD), groups(out[pb:], H, HD)])
        v_g = torch.cat([groups(v.t[:B], H, HD), groups(v.t[pb:], H, HD)])
        qg, kg, batches = torch.cat([qg, qg]), torch.cat([kg, kg]), list(range(B)) + list(range(pb, pb + B))
    else:
        out_g, v_g, batches = groups(out, H, HD), groups(v.t, H, HD), None
    verify(desc, kind, out_g, qg, kg, v_g, scale, dtype, exp2_bound(mask), H, -(-Nk // (64 if pair else 128)),
           batches)

    # batch isolation: the last batch alone (pair: with its two value batches) gives the same bits
    b = B - 1
    alone = Guarded((2 if pair else 1, Nq, C), dtype, dev)
    if pair:
        ops.attention_pair(q.t[b:b + 1], k.t[b:b + 1], v.t[b:b + pb + 1:pb], H, 1, scale, alone.t, variant)
        whole = out[b:b + pb + 1:pb]
    else:
        ops.attention(q.t[b:b + 1], k.t[b:b + 1], v.t[b:b + 1], H, scale, alone.t, variant)
        whole = out[b:b + 1]
    torch.cuda.synchronize()
    alone.check_guard(f"{desc}, batch {b} alone: out")
    assert same_bits(alone.t, whole), f"{desc}: batch {b} alone differs from batch {b} of the full call"
    if pair:   # the same value tensor in both branches gives the same bits in both outputs
        v2 = v.t.clone()
        v2[pb:pb + B] = v2[:B]
        o2 = ops.attention_pair(q.t, k.t, v2, H, pb, scale, None, variant)
        torch.cuda.synchronize()
        assert same_bits(o2[:B], o2[pb:pb + B]), f"{desc}: v[b] == v[b + pair_batches] gives two different outputs"
        assert same_bits(o2[:B], out[:B]), f"{desc}: the first output depends on the second value tensor"


def test_tc_cases_reach_every_compiled_kernel():
    """Without a GPU: the case table launches all 16 attn_tc.cu kernels (4 masks x plain / pair x bf16 / fp16), each
    with the retrieval, uniform and ramp inputs on a multi-block ragged shape."""
    compiled = {(mode, mask, dt) for mode in ("plain", "pair") for mask in MASK_VARIANT for dt in DTYPES}
    reached = {}
    for mode, mask, dt, shape, layout, kind in TC_CASES:
        assert VARIANT_MASK[MASK_VARIANT[mask]] == mask
        if shape[3] > 256 and shape[2] % 128:
            reached.setdefault((mode, mask, dt), set()).add(kind)
    assert len(compiled) == 16 and set(reached) == compiled, sorted(compiled - set(reached))
    assert all(set(REDUCED_KINDS) <= kinds for kinds in reached.values())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("mode", ["plain", "pair"])
def test_variant_aliases_launch_the_same_kernel(cuda_device, mode, dt):
    """Variants 0 and 4 launch the 0xA8 kernel and 1 and 2 the 0x00 kernel: the same bits, which pins the
    variant-to-kernel table the case table relies on; the other masks give different bits."""
    from mvoc_b200 import ops

    dtype, dev = DTYPES[dt], cuda_device
    B, H, Nq, Nk = REDUCED_SHAPE
    q, k, v = (t.to(dev, dtype) for t in make_inputs("random", B, H, Nq, Nk, HD, 2 * B, "cpu", seed=5))
    run = (lambda var: ops.attention_pair(q, k, v, H, B, variant=var)) if mode == "pair" else (
        lambda var: ops.attention(q, k, v[:B], H, variant=var))
    outs = {var: run(var) for var in range(6)}
    torch.cuda.synchronize()
    assert same_bits(outs[0], outs[4]) and same_bits(outs[1], outs[2])
    assert not same_bits(outs[1], outs[4]) and not same_bits(outs[3], outs[4]) and not same_bits(outs[5], outs[4])


# ------------------------------------------------------------------ head_dim 512 and 80
D512_SHAPES = [(2, 1, "both"), (3, 127, "both"), (1, 128, "both"), (2, 129, "both"), (2, 2500, "both"),
               (1, 14080, "fused")]
D512_CASES = [(dt, (B, N), lay, kind) for dt in DTYPES for B, N, lays in D512_SHAPES
              for lay in (LAYOUTS if lays == "both" else (lays,)) for kind in KINDS
              if N < 14080 or dt == "bf16"]
D80_NS = [1, 77, 127, 128, 129, 257, 1024, 4096]
D80_BH = {1: (3, 16), 77: (2, 5), 127: (1, 3), 128: (2, 2), 129: (3, 1), 257: (4, 16), 1024: (1, 4), 4096: (1, 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", D512_CASES, ids=lambda c: f"{c[0]}-{shape_id(c[1])}-{c[2]}-{c[3]}")
def test_attention_d512_vs_float64(cuda_device, case):
    from mvoc_b200 import ops

    dt, (B, N), layout, kind = case
    dtype, dev, D = DTYPES[dt], cuda_device, 512
    scale = D ** -0.5
    desc = f"ops.attention_d512 {dt} mask 0x00 plain, 128-key blocks, B={B} N={N} {layout} {kind}"
    q, k, v = qkv_operands(*make_inputs(kind, B, 1, N, N, D, B, "cpu", seed=N + B), dtype, dev, layout)
    make_out = out_maker((B, N, D), dtype, dev, layout)
    out = run_twice(desc, lambda o: ops.attention_d512(q.t, k.t, v.t, scale, o), make_out, {"q": q, "k": k, "v": v})
    verify(desc, kind, out, q.t, k.t, v.t, scale, dtype, exp2_bound(0), 1, -(-N // 128))
    b = B - 1
    alone = ops.attention_d512(q.t[b:b + 1], k.t[b:b + 1], v.t[b:b + 1], scale)
    torch.cuda.synchronize()
    assert same_bits(alone, out[b:b + 1]), f"{desc}: batch {b} alone differs from batch {b} of the full call"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("N", D80_NS)
@pytest.mark.parametrize("dt", list(DTYPES))
def test_attention_d80_vs_float64(cuda_device, dt, N, layout, kind):
    from mvoc_b200 import ops

    dtype, dev, D = DTYPES[dt], cuda_device, 80
    B, H = D80_BH[N]
    scale = D ** -0.5
    desc = f"ops.attention_d80 {dt} mask 0x00 plain, 128-key blocks, B={B} H={H} N={N} {layout} {kind}"
    q, k, v = qkv_operands(*make_inputs(kind, B, H, N, N, D, B, "cpu", seed=N + H), dtype, dev, layout)
    make_out = out_maker((B, N, H * D), dtype, dev, layout)
    out = run_twice(desc, lambda o: ops.attention_d80(q.t, k.t, v.t, H, scale, o), make_out,
                    {"q": q, "k": k, "v": v})
    verify(desc, kind, groups(out, H, D), groups(q.t, H, D), groups(k.t, H, D), groups(v.t, H, D), scale, dtype,
           exp2_bound(0), H, -(-N // 128))
    b = B - 1
    alone = ops.attention_d80(q.t[b:b + 1], k.t[b:b + 1], v.t[b:b + 1], H, scale)
    torch.cuda.synchronize()
    assert same_bits(alone, out[b:b + 1]), f"{desc}: batch {b} alone differs from batch {b} of the full call"


# ------------------------------------------------------------------ temporal attention (bf16 only)
# (P, T, H): T exact (16, 32) and masked; P * H odd leaves the last CTA of 4 warps partial
TEMPORAL_SHAPES = [(5, 1, 1), (7, 2, 5), (9, 15, 1), (33, 16, 5), (3, 17, 20), (13, 31, 1), (11, 32, 5),
                   (257, 16, 20)]
# (B, T, S, H) of the frames entry: rows in (b, t, pixel) order, read from fused QKV rows
FRAMES_SHAPES = [(1, 1, 7, 5), (2, 2, 5, 1), (1, 15, 9, 5), (2, 16, 33, 5), (1, 17, 3, 20), (2, 31, 5, 1),
                 (1, 32, 11, 5)]


def temporal_kernel(T):
    return f"TP={16 if T <= 16 else 32} {'exact' if T in (16, 32) else 'masked'}"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("shape", TEMPORAL_SHAPES, ids=shape_id)
def test_temporal_attention_vs_float64(cuda_device, shape, layout, kind):
    from mvoc_b200 import ops

    P, T, H = shape
    dtype, dev, scale = torch.bfloat16, cuda_device, HD ** -0.5
    desc = f"ops.temporal_attention bf16 exp2f {temporal_kernel(T)}, P={P} T={T} H={H} {layout} {kind}"
    q, k, v = qkv_operands(*make_inputs(kind, P, H, T, T, HD, P, "cpu", seed=P + T + H), dtype, dev, layout)
    make_out = out_maker((P, T, H * HD), dtype, dev, layout)
    out = run_twice(desc, lambda o: ops.temporal_attention(q.t, k.t, v.t, H, scale, o), make_out,
                    {"q": q, "k": k, "v": v})
    verify(desc, kind, groups(out, H, HD), groups(q.t, H, HD), groups(k.t, H, HD), groups(v.t, H, HD), scale, dtype,
           exp2_bound(0), H, 1)
    alone = ops.temporal_attention(q.t[P - 1:], k.t[P - 1:], v.t[P - 1:], H, scale)
    torch.cuda.synchronize()
    assert same_bits(alone, out[P - 1:]), f"{desc}: problem {P - 1} alone differs from the full call"


def frames_rows(t, B, T, S):
    """[B*S, T, C] problems -> [B*T*S, C] rows in (b, t, pixel) order, and back."""
    return t.reshape(B, S, T, -1).permute(0, 2, 1, 3).reshape(B * T * S, -1)


def frames_problems(t, B, T, S):
    return t.reshape(B, T, S, -1).permute(0, 2, 1, 3).reshape(B * S, T, -1)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", FRAMES_SHAPES, ids=shape_id)
def test_temporal_attention_frames_vs_float64(cuda_device, shape, kind):
    from mvoc_b200 import ops

    B, T, S, H = shape
    dtype, dev, scale, C = torch.bfloat16, cuda_device, HD ** -0.5, H * HD
    rows = B * T * S
    desc = f"ops.temporal_attention_frames bf16 exp2f {temporal_kernel(T)}, B={B} T={T} S={S} H={H} fused {kind}"
    q, k, v = (Guarded((rows, C), dtype, dev, ld=3 * C, fill=frames_rows(t, B, T, S))
               for t in make_inputs(kind, B * S, H, T, T, HD, B * S, "cpu", seed=rows + H))
    make_out = lambda: Guarded((rows, C), dtype, dev, ld=C + 64)
    out = run_twice(desc, lambda o: ops.temporal_attention_frames(q.t, k.t, v.t, H, B, T, S, scale, o), make_out,
                    {"q": q, "k": k, "v": v})
    pg = lambda t: groups(frames_problems(t, B, T, S), H, HD)
    verify(desc, kind, pg(out), pg(q.t), pg(k.t), pg(v.t), scale, dtype, exp2_bound(0), H, 1)
    n = T * S
    alone = ops.temporal_attention_frames(q.t[-n:], k.t[-n:], v.t[-n:], H, 1, T, S, scale)
    torch.cuda.synchronize()
    assert same_bits(alone, out[-n:]), f"{desc}: video {B - 1} alone differs from the full call"


# ------------------------------------------------------------------ the injected attention entry
INJECT_CASES = [(mode, dt, px, kind) for px in (880, 4096) for mode in ("spatial_shared", "spatial", "temporal")
                for dt in DTYPES for kind in ("random", "uniform", "ramp") if mode != "temporal" or dt == "bf16"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", INJECT_CASES, ids=lambda c: f"{c[0]}-{c[1]}-px{c[2]}-{c[3]}")
def test_attention_inject_vs_float64(cuda_device, case):
    """Float64 attention of the q and k the entry left blended in place (test_kernels_gpu checks those against the
    blend kernel); with the shared softmax the cond branch uses the uncond branch's blended q and k."""
    from mvoc_b200 import ops

    mode, dt, px, kind = case
    dtype, dev, scale = DTYPES[dt], cuda_device, HD ** -0.5
    n_obj, frames, H = 2, 2, 2
    nb, C = n_obj + 3, H * HD
    temporal, share = mode == "temporal", mode == "spatial_shared"
    desc = (f"ops.attention_inject_ {dt} {'exp2f' if temporal else 'mask 0xa8'} {mode}, n_obj={n_obj} "
            f"frames={frames} pixels={px} fused {kind}")
    if temporal:   # problems (branch, pixel) over frames, stored in (branch, frame, pixel) rows
        src = make_inputs(kind, nb * px, H, frames, frames, HD, nb * px, "cpu", seed=px + 1)
        src = [t.reshape(nb, px, frames, C).permute(0, 2, 1, 3).reshape(nb * frames, px, C) for t in src]
    else:
        src = make_inputs(kind, nb * frames, H, px, px, HD, nb * frames, "cpu", seed=px)
    q, k, v = qkv_operands(*src, dtype, dev, "fused")
    mask = (torch.rand(n_obj, frames * px, generator=torch.Generator().manual_seed(px)) < 0.4).to(torch.uint8).to(dev)
    outs, blended = [], []
    for _ in range(2):
        for g in (q, k):
            g.buf.view(torch.int16).copy_(g.snapshot)
        o = Guarded((nb * frames, px, C), dtype, dev, ld=C + 64)
        ops.attention_inject_(q.t, k.t, v.t, mask, H, n_obj, frames, True, temporal, scale, o.t, 0,
                              share if not temporal else None)
        torch.cuda.synchronize()
        o.check_guard(f"{desc}: out")
        outs.append(o.t)
        blended.append((q.t.clone(), k.t.clone()))
    v.check_unchanged(f"{desc}: v")
    q.check_guard(f"{desc}: q")
    k.check_guard(f"{desc}: k")
    assert same_bits(outs[0], outs[1]) and same_bits(blended[0][0], blended[1][0]) and \
        same_bits(blended[0][1], blended[1][1]), f"{desc}: two identical calls gave different bits"
    out, qb, kb = outs[0], q.t, k.t
    if share:       # the blend wrote the composites' q', k' once, into the uncond slot
        qb, kb = qb.clone(), kb.clone()
        cond, uncond = slice((nb - 1) * frames, nb * frames), slice((nb - 2) * frames, (nb - 1) * frames)
        qb[cond], kb[cond] = qb[uncond], kb[uncond]
    if temporal:
        pg = lambda t: groups(t.reshape(nb, frames, px, C).permute(0, 2, 1, 3).reshape(nb * px, frames, C), H, HD)
        nkb = 1
    else:
        pg, nkb = (lambda t: groups(t, H, HD)), -(-px // 128)
    verify(desc, kind, pg(out), pg(qb), pg(kb), pg(v.t), scale, dtype, exp2_bound(0 if temporal else 0xA8), H, nkb)


# ------------------------------------------------------------------ wrapper checks (CUDA tensors, no launch)
@pytest.mark.gpu
def test_attention_wrappers_reject_bad_operands_before_launch(cuda_device):
    """Every attention wrapper refuses, before any launch: operands of different dtypes, an out that is not the shape
    the kernel writes, and an out whose last dimension is not contiguous; attention_pair also pair_batches < B.  The
    temporal kernel is bf16-only: an fp16 call fails in the C entry, also before the launch."""
    from mvoc_b200 import _cabi, ops

    dev, bf, fp = cuda_device, torch.bfloat16, torch.float16
    z = lambda *s, dt=bf: torch.zeros(*s, dtype=dt, device=dev)
    x, C = z(2, 128, 128), 128

    def bad_out(shape, dt=bf):
        return [z(*shape, dt=fp if dt == bf else bf), z(shape[0] + 1, *shape[1:], dt=dt),
                z(*shape[:-2], shape[-2] - 1, shape[-1], dt=dt), z(*shape[:-1], 2 * shape[-1], dt=dt)[..., ::2],
                z(*shape, dt=torch.float32)]

    calls = {
        "attention": (lambda q, k, v, o: ops.attention(q, k, v, 2, out=o), (x, x, x), (2, 128, C)),
        "attention_pair": (lambda q, k, v, o: ops.attention_pair(q, k, v, 2, 2, out=o), (x, x, z(4, 128, C)),
                           (4, 128, C)),
        "attention_d512": (lambda q, k, v, o: ops.attention_d512(q, k, v, out=o), (z(2, 64, 512),) * 3, (2, 64, 512)),
        "attention_d80": (lambda q, k, v, o: ops.attention_d80(q, k, v, 2, out=o), (z(2, 64, 160),) * 3, (2, 64, 160)),
        "temporal_attention": (lambda q, k, v, o: ops.temporal_attention(q, k, v, 2, out=o), (z(8, 16, C),) * 3,
                               (8, 16, C)),
        "temporal_attention_frames": (lambda q, k, v, o: ops.temporal_attention_frames(q, k, v, 2, 1, 4, 8, out=o),
                                      (z(32, C),) * 3, (32, C)),
        "attention_inject_": (lambda q, k, v, o: ops.attention_inject_(
            q, k, v, z(2, 2 * 64, dt=torch.uint8), 2, 2, 2, True, False, out=o), (z(10, 64, C),) * 3, (10, 64, C)),
    }
    for name, (call, (q, k, v), shape) in calls.items():
        for o in bad_out(shape):
            with pytest.raises(ValueError, match=name):
                call(q, k, v, o)
        for i in range(3):
            qkv = [q, k, v]
            qkv[i] = qkv[i].to(fp)
            with pytest.raises(ValueError, match=name):
                call(*qkv, z(*shape))
    for pb in (1, 2):
        with pytest.raises(ValueError, match="attention_pair"):
            ops.attention_pair(z(3, 128, C), z(3, 128, C), z(3 + pb, 128, C), 2, pb)
    t16 = z(8, 16, C, dt=fp)
    with pytest.raises(_cabi.MvocError, match="bf16 only"):
        ops.temporal_attention(t16, t16, t16, 2)
    torch.cuda.synchronize()
