"""Every compiled configuration of the tcgen05 GEMM kernel (csrc/gemm_tc.cu) element by element against float64.

The kernel is compiled 28 times: the linear epilogue at tile widths BN 256, 192, 160, 128 and 64 and the GEGLU epilogue
at 256 and 128, each on one CTA and as a CTA pair, each in bf16 and fp16.  The Linear entries run every one of them
(forced by `variant = BN << 8 | pair`, with the tile plan checked before the launch, since pairs can only be allowed);
the convolution entries run the row boxes production shapes pick, degenerate images whose box is wider than the grid,
the second K source, and the stride-2 tap origins at every edge.

Every operand is a view into a NaN-filled allocation, so a read of memory beside an operand (instead of TMA zero fill)
makes a NaN output, and a write beside the output overwrites a NaN.  Each output element must satisfy

    |out - ref| <= u |ref| + 2^-16 S,      S = |x| |w|^T + |b| + |r|  (the same sum over absolute values)

where ref and S are float64 from the same 16-bit inputs and u is the unit roundoff of the output type: the first term is
the single rounding of the fp32 accumulator, the second an allowance for fp32 accumulation that stays far below the
error of a wrong tap, a missing K chunk or a missing bias.  A failure names the kernel, the row box and the worst
element with its row and column tile.  Every case runs twice and must give the same bits (the epilogue's staging
buffers are reused while TMA stores still read them)."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

from mvoc_b200 import _cabi

B200_SMS = 148
GUARD = 2048                                   # NaN elements before and after every operand (keeps 16-byte alignment)
UNIT = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
ACC = 2.0 ** -16                               # fp32 accumulation allowance, relative to S
GELU_SLOPE = 1.13                              # max |gelu'(x)| = 1.129 at x = sqrt 2
ERF_ERR = 1e-6                                 # GEGLU epilogue's erf (Abramowitz-Stegun 7.1.26), relative to |value|
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
WIDTHS = {"linear": (256, 192, 160, 128, 64), "geglu": (256, 128)}


def gemm_plan(rows, n, geglu, variant, sms):
    """(BN, CTA pair, tail columns) that the GEMM entries launch for a Linear of `rows` rows (host logic only)."""
    lib = _cabi.load()
    bn, pair, tail = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _cabi.check(lib.mvoc_gemm_plan(rows, n, int(geglu), variant, sms, ctypes.byref(bn), ctypes.byref(pair),
                                   ctypes.byref(tail)), "mvoc_gemm_plan")
    return bn.value, bool(pair.value), tail.value


def choose_box(d1, d2, d3):
    """gemm_tc.cu's choose_box: the power-of-two row box (b1, b2, b3), b1 b2 b3 = 128, that pads the (d1, d2, d3)
    grid least; ties go to the widest b1."""
    best, box = None, None
    for w in (128, 64, 32, 16, 8, 4, 2, 1):
        h = 128 // w
        while h >= 1:
            n = 128 // (w * h)
            padded = -(-d1 // w) * w * -(-d2 // h) * h * -(-d3 // n) * n
            if best is None or padded < best:
                best, box = padded, (w, h, n)
            h //= 2
    return box


# ------------------------------------------------------------------ harness
class Guarded:
    """A tensor of `shape` inside a NaN-filled allocation: GUARD NaNs before and after it and, when ld > shape[-1],
    ld - shape[-1] NaN columns after each row (a column slice with row stride ld)."""

    def __init__(self, shape, dtype, device, ld=None, fill=None):
        cols, rows = shape[-1], math.prod(shape[:-1])
        ld = ld or cols
        self.buf = torch.full((2 * GUARD + rows * ld,), float("nan"), dtype=dtype, device=device)
        self.t = self.buf[GUARD:GUARD + rows * ld].view(rows, ld)[:, :cols].view(shape)
        self.guard = torch.ones(self.buf.numel(), dtype=torch.bool, device=device)
        self.guard[GUARD:GUARD + rows * ld].view(rows, ld)[:, :cols] = False
        if fill is not None:
            self.t.copy_(fill)
        self.snapshot = self.buf.view(torch.int16).clone()

    def check_guard(self, what):
        nan = torch.tensor(float("nan"), dtype=self.buf.dtype).view(torch.int16).item()
        bad = (self.guard & (self.buf.view(torch.int16) != nan)).nonzero()
        assert bad.numel() == 0, (f"{what}: {bad.numel()} guard elements overwritten, the first at allocation "
                                  f"element {int(bad[0])} (the tensor starts at {GUARD})")

    def check_unchanged(self, what):
        assert torch.equal(self.buf.view(torch.int16), self.snapshot), f"{what}: an input (or its guard) was written"


def operand(shape, dtype, device, scale=1.0, ld=None):
    return Guarded(shape, dtype, device, ld=ld, fill=torch.randn(shape, device=device) * scale)


class Kernel:
    """What one launch runs: entry, dtype, tile width, CTA mode and row box, for failure messages."""

    def __init__(self, entry, dtype, grid, n, variant, sms, geglu=False):
        self.entry, self.dtype, self.geglu = entry, dtype, geglu
        self.box = (128, 1, 1) if entry.startswith("mvoc_linear") else choose_box(*grid)
        m_tiles = math.prod(-(-d // b) for d, b in zip(grid, self.box))
        self.bn, self.pair, self.tail = gemm_plan(128 * m_tiles, n, geglu, variant, sms)
        self.out_cols = self.bn // 2 if geglu else self.bn

    def __str__(self):
        return (f"{self.entry} {str(self.dtype)[6:]} BN={self.bn} {'CTA pair' if self.pair else 'one CTA'} "
                f"box={self.box}")


def check_bound(kernel, out, ref, bound):
    """out, ref, bound: [d3, d2, d1, C] (the row grid of the kernel, outermost first).  Returns the largest
    err / bound, and the largest (err - half an ulp of out) / (bound - u |ref|): a lower bound on the share of the
    accumulation allowance the kernel used (informational: the rounding term alone brings err / bound close to 1)."""
    out = out.double()
    finite = torch.isfinite(out)
    if not bool(finite.all()):
        d3, d2, d1, c = (int(i) for i in (~finite).nonzero()[0])
        raise AssertionError(f"{kernel}: {int((~finite).sum())} outputs are not finite (a read beside an operand or "
                             f"an unwritten tile), the first at row (d1, d2, d3) = {(d1, d2, d3)} column {c}")
    ratio = (out - ref).abs() / bound.clamp_min(torch.finfo(torch.float64).tiny)
    worst = int(ratio.argmax())
    r = float(ratio.view(-1)[worst])
    if r > 1.0:
        idx = []
        for size in reversed(ratio.shape):
            idx.append(worst % size)
            worst //= size
        c, d1, d2, d3 = idx
        b1, b2, b3 = kernel.box
        raise AssertionError(
            f"{kernel}: worst element at row (d1, d2, d3) = {(d1, d2, d3)} column {c}, in row tile "
            f"{(d1 // b1, d2 // b2, d3 // b3)} and column tile {c // kernel.out_cols}: out {float(out[d3, d2, d1, c]):.6g}"
            f" ref {float(ref[d3, d2, d1, c]):.6g} bound {float(bound[d3, d2, d1, c]):.3g}, err / bound = {r:.3g}")
    precision = 8 if kernel.dtype == torch.bfloat16 else 11
    half_ulp = torch.ldexp(torch.ones_like(out), torch.frexp(out).exponent - precision - 1).clamp_min(2.0 ** -25)
    allowance = bound - UNIT[kernel.dtype] * ref.abs()
    acc = float(((out - ref).abs() - half_ulp).clamp_min(0).div(allowance).max())
    return r, acc


def run_twice(kernel, launch, make_out, inputs):
    """Launch into two fresh NaN-guarded outputs; check guards, inputs and that both calls gave the same bits."""
    outs = []
    for _ in range(2):
        out = make_out()
        launch(out.t)
        outs.append(out)
    torch.cuda.synchronize()
    for name, g in inputs.items():
        if g is not None:
            g.check_unchanged(f"{kernel}: {name}")
    for o in outs:
        o.check_guard(f"{kernel}: out")
    assert torch.equal(outs[0].t.contiguous().view(torch.int16), outs[1].t.contiguous().view(torch.int16)), (
        f"{kernel}: two identical calls gave different outputs")
    return outs[0].t


def tensor(g):
    return None if g is None else g.t


def linear_terms(x, w, b=None, r=None):
    """float64 ref and magnitude S of x w^T (+ b) (+ r) from the 16-bit operands."""
    x, w = x.double(), w.double()
    b = None if b is None else b.double()
    ref, mag = F.linear(x, w, b), F.linear(x.abs(), w.abs(), None if b is None else b.abs())
    if r is not None:
        ref, mag = ref + r.double(), mag + r.double().abs()
    return ref, mag


def geglu_reference(x, w, b, dtype):
    """value * gelu(gate) with value and gate in float64, and its bound: each half's accumulation allowance goes
    through the product."""
    ref, mag = linear_terms(x, w, b)
    v, g = ref.chunk(2, dim=-1)
    mv, mg = mag.chunk(2, dim=-1)
    gelu = F.gelu(g)
    ref = v * gelu
    bound = UNIT[dtype] * ref.abs() + ACC * mv * gelu.abs() + v.abs() * (GELU_SLOPE * ACC * mg + ERF_ERR)
    return ref, bound


# ------------------------------------------------------------------ every kernel, through the Linear entries
# (epilogue, BN) -> N (GEGLU: F) of the case: a narrower tail tile wherever the width allows one.  160 cannot have a
# tail (tails are multiples of 64) and N must be a multiple of 64, so 160 gets four full tiles; GEGLU never has a tail.
LINEAR_N = {("linear", 256): 320, ("linear", 192): 448, ("linear", 160): 640, ("linear", 128): 320,
            ("linear", 64): 320, ("geglu", 256): 384, ("geglu", 128): 192}
LONG_K, SHORT_K = 576, 64      # 9 K chunks: one more than the deepest shared-memory ring (8 stages)
LINEAR_CASES = [(epi, bn, pair, dt, shape) for (epi, bn) in LINEAR_N for pair in (False, True) for dt in DTYPES
                for shape in ("long", "m1", "m129")]


def linear_id(case):
    epi, bn, pair, dt, shape = case
    return f"{epi}-bn{bn}-{'pair' if pair else 'one_cta'}-{dt}-{shape}"


def linear_dims(epi, bn, shape, sms):
    """(M, K, N, bias and residual on).  The long shape has an odd number of row tiles (the last CTA pair runs the
    padding tile) in at least two waves (both TMEM accumulator buffers are reused), the last tile partial; the short
    shapes are one row, and 129 rows (one pair whose second tile is the padding tile)."""
    n = LINEAR_N[(epi, bn)]
    if shape == "long":
        n_tiles = -(-n // (bn // 2 if epi == "geglu" else bn))
        return 128 * (2 * -(-sms // n_tiles) + 1) - 37, LONG_K, n, True
    return {"m1": 1, "m129": 129}[shape], SHORT_K, n, False


def run_linear(dev, epi, bn, pair, dtype, M, K, N, extras, sms):
    """One Linear / GEGLU launch on guarded operands with the kernel forced: (kernel, out, operands)."""
    from mvoc_b200 import ops

    geglu = epi == "geglu"
    variant = bn << 8 | int(pair)
    kernel = Kernel("mvoc_linear_geglu" if geglu else "mvoc_linear", dtype, (M, 1, 1), N, variant, sms, geglu)
    assert (kernel.bn, kernel.pair, kernel.tail) == (bn, pair, N % kernel.out_cols), (
        f"the plan does not launch the kernel this case names: {kernel}, tail {kernel.tail}")
    w_rows = 2 * N if geglu else N
    w = operand((w_rows, K), dtype, dev, K ** -0.5)
    b = operand((w_rows,), dtype, dev) if extras else None
    if geglu:
        x, r = operand((M, K), dtype, dev), None
        make_out = lambda: Guarded((M, N), dtype, dev)
        launch = lambda o: ops.linear_geglu(x.t, w.t, tensor(b), out=o, variant=variant)
    else:
        x = operand((M, K), dtype, dev, ld=K + 64)
        r = operand((M, N), dtype, dev, ld=N + 32) if extras else None
        make_out = lambda: Guarded((M, N), dtype, dev, ld=N + 96)
        launch = lambda o: ops.linear(x.t, w.t, tensor(b), tensor(r), out=o, variant=variant)
    operands = {"x": x, "w": w, "bias": b, "residual": r}
    return kernel, run_twice(kernel, launch, make_out, operands), operands


def device_sms(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


@pytest.mark.gpu
@pytest.mark.parametrize("case", LINEAR_CASES, ids=linear_id)
def test_every_kernel_vs_float64(cuda_device, case):
    epi, bn, pair, dt, shape = case
    sms = device_sms(cuda_device)
    M, K, N, extras = linear_dims(epi, bn, shape, sms)
    torch.manual_seed(M + K + N + bn)
    dtype = DTYPES[dt]
    kernel, out, operands = run_linear(cuda_device, epi, bn, pair, dtype, M, K, N, extras, sms)
    x, w, b, r = (tensor(operands[k]) for k in ("x", "w", "bias", "residual"))
    if epi == "geglu":
        ref, bound = geglu_reference(x, w, b, dtype)
    else:
        ref, mag = linear_terms(x, w, b, r)
        bound = UNIT[dtype] * ref.abs() + ACC * mag
    ratio, acc = check_bound(kernel, out.view(1, 1, M, N), ref.view(1, 1, M, N), bound.view(1, 1, M, N))
    print(f"max err/bound {ratio:.4f} accumulation share {acc:.4f}")


def test_linear_cases_reach_every_compiled_kernel():
    """Without a GPU: on a 148-SM B200 the case table above launches all 28 compiled kernels, each with the tail tile
    its width allows; and the row boxes in the convolution table below are the ones choose_box picks."""
    reached = set()
    for epi, bn, pair, dt, shape in LINEAR_CASES:
        M, K, N, _ = linear_dims(epi, bn, shape, B200_SMS)
        out_cols = bn // 2 if epi == "geglu" else bn
        assert gemm_plan(M, N, epi == "geglu", bn << 8 | int(pair), B200_SMS) == (bn, pair, N % out_cols), \
            linear_id((epi, bn, pair, dt, shape))
        reached.add((epi, bn, pair, dt))
    compiled = {(epi, bn, pair, dt) for epi, widths in WIDTHS.items() for bn in widths for pair in (False, True)
                for dt in DTYPES}
    assert len(compiled) == 28 and reached == compiled, sorted(compiled - reached)
    assert {bn for (epi, bn), n in LINEAR_N.items() if epi == "linear" and n % bn} == {256, 192, 128}
    for entry, dims, pads, box, _ in CONV_CASES:
        assert choose_box(*conv_grid(entry, dims, pads)) == box, (entry, dims, pads)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("epi", ["linear", "geglu"])
def test_tilings_are_bit_identical(cuda_device, epi, dt):
    """Each output element sums its K terms in the same order whatever the tile width and CTA mode (only the rows
    and columns a tile covers change), so every kernel of one epilogue gives the same bits for one problem."""
    sms = device_sms(cuda_device)
    N = 320 if epi == "linear" else 384       # every width tiles it (192 with a 128-wide tail)
    M = 128 * (2 * -(-sms // 2) + 1) - 37
    outs = {}
    for bn in WIDTHS[epi]:
        for pair in (False, True):
            torch.manual_seed(7)                # the same operands for every kernel
            outs[(bn, pair)] = run_linear(cuda_device, epi, bn, pair, DTYPES[dt], M, LONG_K, N, True, sms)[1]
    base_key = next(iter(outs))
    base = outs[base_key].contiguous()
    diffs = []
    for (bn, pair), o in outs.items():
        o = o.contiguous()
        if not torch.equal(o.view(torch.int16), base.view(torch.int16)):
            d = (o.double() - base.double()).abs()
            diffs.append(f"BN={bn} {'pair' if pair else 'one CTA'}: {int((d > 0).sum())} elements differ, max "
                         f"{float(d.max()):.3g}")
    assert not diffs, f"against BN={base_key[0]} one CTA: " + "; ".join(diffs)


# ------------------------------------------------------------------ row boxes and sources, through the convolutions
CIN, COUT, CIN2 = 64, 192, 128
# entry, dims (conv3x3 and stride 2: input W x H x N; temporal: S x T x B), stride-2 pads, the row box choose_box gives
# on the row grid (the output grid), and why the case is here
CONV_CASES = [
    ("conv3x3", (160, 88, 3), None, (32, 4, 1), "config 5 level 0"),
    ("conv3x3", (80, 44, 10), None, (16, 4, 2), "config 5 level 1"),
    ("conv3x3", (40, 22, 80), None, (8, 2, 8), "config 5 level 2"),
    ("conv3x3", (20, 11, 80), None, (4, 4, 8), "config 5 level 3"),
    ("conv3x3", (8, 8, 9), None, (8, 8, 2), "config 2 level 3; frames not a multiple of b3"),
    ("conv3x3", (300, 1, 1), None, (128, 1, 1), "one-row image"),
    ("conv3x3", (1, 1, 200), None, (1, 1, 128), "1x1 images: box wider than the grid"),
    ("conv3x3", (1, 1, 3), None, (32, 1, 4), "1x1 images: box wider than the grid"),
    ("conv3x3", (7, 1, 5), None, (16, 1, 8), "box wider than the grid"),
    ("conv3x3", (1, 7, 5), None, (2, 8, 8), "box wider than the grid"),
    ("temporal", (256, 16, 2), None, (128, 1, 1), "video edges: first and last frames see zeros"),
    ("temporal", (100, 8, 3), None, (16, 8, 1), "video edges inside one box"),
    ("temporal", (8, 32, 5), None, (8, 16, 1), "video edges inside one box"),
    ("temporal", (256, 1, 1), None, (128, 1, 1), "one frame: both outer taps are padding"),
    ("temporal", (4096, 2, 5), None, (128, 1, 1), "two frames"),
    ("conv3x3_s2", (80, 44, 80), (0, 1), (8, 2, 8), "VAE downsampler padding, config 5 level 2"),
    ("conv3x3_s2", (80, 44, 80), (1, 1), (8, 2, 8), "torch padding=1"),
    ("conv3x3_s2", (77, 45, 3), (0, 1), (16, 8, 1), "odd extents"),
    ("conv3x3_s2", (2, 2, 7), (0, 1), (16, 1, 8), "one output pixel: box wider than the grid"),
]
CONV_VARIANTS = {"one_cta": 0, "pairs": 1, "bn64_pairs": 64 << 8 | 1}


def conv_id(case):
    entry, dims, pads, _, _ = case
    return f"{entry}-{'x'.join(map(str, dims))}" + (f"-pad{pads[0]}{pads[1]}" if pads else "")


def conv_grid(entry, dims, pads):
    """The (d1, d2, d3) row grid of the kernel: the output pixels (W, H, N) or (S, T, B)."""
    if entry != "conv3x3_s2":
        return dims
    W, H, N = dims
    return tuple((n + pads[0] + pads[1] - 3) // 2 + 1 for n in (W, H)) + (N,)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", CONV_VARIANTS)
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("case", CONV_CASES, ids=conv_id)
def test_conv_row_boxes_vs_float64(cuda_device, case, dt, variant):
    from mvoc_b200 import ops

    entry, dims, pads, _, _ = case
    dtype, v, dev = DTYPES[dt], CONV_VARIANTS[variant], cuda_device
    grid = conv_grid(entry, dims, pads)
    kernel = Kernel("mvoc_" + {"conv3x3": "conv3x3_nhwc", "temporal": "temporal_conv3",
                               "conv3x3_s2": "conv3x3_s2_nhwc"}[entry], dtype, grid, COUT, v, device_sms(dev))
    torch.manual_seed(sum(dims) + v)
    d1, d2, d3 = grid
    b = operand((COUT,), dtype, dev)
    if entry == "temporal":
        S, T, B = dims
        x = operand((B * T, S, CIN), dtype, dev)
        w = (torch.randn(COUT, CIN, 3, 1, 1, device=dev) * (3 * CIN) ** -0.5).to(dtype)
        wt = Guarded((3, COUT, CIN), dtype, dev, fill=ops.conv_taps(w))
        r = operand((B * T, S, COUT), dtype, dev)
        inputs = {"x": x, "w": wt, "bias": b, "residual": r}
        make_out = lambda: Guarded((B * T, S, COUT), dtype, dev)
        launch = lambda o: ops.temporal_conv3(x.t, wt.t, b.t, B, T, r.t, out=o, variant=v)
        x5 = x.t.double().view(B, T, S, CIN).permute(0, 3, 1, 2)[..., None]        # [B, Cin, T, S, 1]
        conv = lambda xx, ww, bb: F.conv3d(xx, ww, bb, padding=(1, 0, 0))[..., 0].permute(0, 2, 3, 1)
        ref, mag = conv(x5, w.double(), b.t.double()), conv(x5.abs(), w.double().abs(), b.t.double().abs())
        ref, mag = ref + r.t.double().view(ref.shape), mag + r.t.double().abs().view(ref.shape)
    else:
        W, H, N = dims
        x = operand((N, H, W, CIN), dtype, dev)
        w = (torch.randn(COUT, CIN, 3, 3, device=dev) * (9 * CIN) ** -0.5).to(dtype)
        wt = Guarded((9, COUT, CIN), dtype, dev, fill=ops.conv_taps(w))
        xc = x.t.double().permute(0, 3, 1, 2)
        if entry == "conv3x3":
            x2 = operand((N, H, W, CIN2), dtype, dev)
            w2 = operand((COUT, CIN2), dtype, dev, CIN2 ** -0.5)
            r = operand((N, H, W, COUT), dtype, dev)
            inputs = {"x": x, "w": wt, "bias": b, "x2": x2, "w2": w2, "residual": r}
            make_out = lambda: Guarded((N, H, W, COUT), dtype, dev)
            launch = lambda o: ops.conv3x3(x.t, wt.t, b.t, r.t, x2.t, w2.t, out=o, variant=v)
            conv = lambda xx, ww, bb: F.conv2d(xx, ww, bb, padding=1).permute(0, 2, 3, 1)
            ref, mag = conv(xc, w.double(), b.t.double()), conv(xc.abs(), w.double().abs(), b.t.double().abs())
            sc, msc = linear_terms(x2.t, w2.t, None, r.t)                 # 1x1 shortcut + residual
            ref, mag = ref + sc, mag + msc
        else:
            pb, pe = pads
            inputs = {"x": x, "w": wt, "bias": b}
            make_out = lambda: Guarded((N, d2, d1, COUT), dtype, dev)
            launch = lambda o: ops.conv3x3_s2(x.t, wt.t, b.t, pad=pads, out=o, variant=v)
            conv = lambda xx, ww, bb: F.conv2d(F.pad(xx, (pb, pe, pb, pe)), ww, bb, stride=2).permute(0, 2, 3, 1)
            ref, mag = conv(xc, w.double(), b.t.double()), conv(xc.abs(), w.double().abs(), b.t.double().abs())
    out = run_twice(kernel, launch, make_out, inputs)
    bound = UNIT[dtype] * ref.abs() + ACC * mag
    shape4 = (d3, d2, d1, COUT)
    ratio, acc = check_bound(kernel, out.reshape(shape4), ref.reshape(shape4), bound.reshape(shape4))
    print(f"max err/bound {ratio:.4f} accumulation share {acc:.4f}")
