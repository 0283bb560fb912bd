"""Float64 references and per-element error bounds for every contraction launch of the train step and the Inception
scorer, and a context manager that checks each such call at the moment it is made.

References work on the packed operands the kernels receive (ops.pack_shapes), so a packed weight that differs from the
fp32 master (UPCONV's pre-summed taps, rounded to bf16 once) is not counted as a kernel error. Every kind is a sum of
per-tap float64 GEMMs over shifted views of the input; dgrad and wgrad are the vector-Jacobian products of the fprop
reference, with wpkT mapped back to the wpk layout (inverse of ops.pack_transpose / tools/probe_conv.py:pack_ref).

Error bounds. r is the float64 result, m the same contraction on absolute values (m >= |r|, one more GEMM per tap).

* Products: bf16 x bf16 is exact in fp32, so the only kernel rounding before the output is in the fp32 accumulation.
  tcgen05.mma adds 16 products (K = 16 per instruction for bf16) into the fp32 accumulator, once per instruction; a
  split-K launch adds its split partials in fp32, a bias or an accumulate-into buffer adds one more fp32 add. The chain
  behind one output therefore has n = ceil(K / 16) + splits + 2 rounding steps (2: bias / existing accumulator and the
  final store), each with relative error at most U_ACC = 2^-23 (one unit in the last place: this allows an accumulator
  that truncates rather than rounds to nearest).
* The deterministic worst case, n * U_ACC * m, grows linearly with K and would hide every fault at production sizes
  (at K = 18 432 it is 2^-12.8 m; for a 1.6 M-pixel wgrad it is 2^-6.4 m). The bound used instead is Higham and Mary's
  probabilistic one (SIAM J. Sci. Comput. 41(5), 2019, Thm. 2.4): with the step errors independent and mean zero,
  |acc - r| <= gamma(n) * m, gamma(n) = exp(LAMBDA * sqrt(n) * U_ACC + n * U_ACC^2 / (1 - U_ACC)) - 1, with probability
  at least 1 - 2 n exp(-LAMBDA^2 (1 - U_ACC)^2 / 2) per element. LAMBDA = 10 makes that 4e-22 * n: over the ~1e10
  elements and n <= 1e5 steps of the GPU tests, a false alarm has probability below 1e-6. A truncating accumulator
  breaks the mean-zero assumption by a bias of at most n * U_ACC / 2 * (sum of the partial sums); for zero-mean data
  the partial sums are ~ sqrt(K) |a||b|, not K |a||b|, which keeps that bias below 1 % of gamma(n) m at K = 18 432.
  For K = 18 432 (n = 1155): gamma = 2^-13.6, so c = gamma ~ the 2^-14 one would guess, derived rather than assumed.
* bf16 output (round to nearest, unit roundoff 2^-8): |got - r| <= 2^-8 |r| + (1 + 2^-8) gamma(n) m.
  LeakyReLU / ReLU in the epilogue are 1-Lipschitz and applied to both sides; the bf16 term uses |act(r)|.
  A dgrad epilogue operand src (EPI_ADD: r + src; EPI_LRELU_MASK: r * (src > 0 ? 1 : 0.2)) may be applied after a
  separate bf16 rounding of the convolution (ops._epi_apply): one more 2^-8 (1 + 2^-8) |conv| term, scaled by the mask.
* fp32-accurate mode (3-way bf16 split, six plane products, fp32 result): the split of x and of the packed weight is
  exact to 2^-24 relative, the three dropped plane products (mid*lo, lo*mid, lo*lo) are below 2.1 * 2^-24 |a||b|:
  |got - r| <= (2^-22 + gamma(n + 6)) m, with r computed from the fp32 x and the sum of the weight planes.
* BatchNorm statistics (per group and channel, the change of the fp64 slot across the call) against float64 sums of
  the returned tensor: per-block partials are fp32 sums (U32 = 2^-24, round to nearest) of at most the group's rows,
  combined with fp64 atomics: |got - S1| <= gamma_U32(rows) sum|y|, |got - S2| <= gamma_U32(rows) sum y^2. fp32 outputs
  (fp32-accurate mode) are summed in fp64: the same with U = 2^-52.
* Linears (fp32 operands, fp32 accumulation; bf16 dy is exact in fp32): |got - r| <= gamma(K + 64) m, plus the bf16 term
  when the output is bf16 (the + 64 covers the partial slabs of linear_bwd_x).

Sensitivity (tests/test_launch_ref_host.py). At the step's largest fprop / dgrad contraction (K = 9 x 2048) the bound is
2^-8 |r| + 2^-13.6 m: one dropped border tap (2048 products) and one 16-channel K block dropped from a 128-row tile
exceed it. wgrad at 24 * 256^2 = 1.57 M pixels: gamma(98 306) = 2^-11.7, about 400 for unit-variance operands, while a
128-pixel tile contributes ~ sqrt(128) = 11 per element: a single dropped tile of zero-mean data is below the bound.
The smallest dropped run the bound catches there is 256 tiles (32 768 pixels, 2 % of the pixels: the largest of the 256
per-element sums then exceeds the bound with near certainty); at 8192 pixels one dropped tile is caught.
"""
import json
import math
import os
from contextlib import contextmanager

import torch

CONV3, UPCONV, CONV4S2, GEMM = 0, 1, 2, 3
KIND_NAMES = {CONV3: "CONV3", UPCONV: "UPCONV", CONV4S2: "CONV4S2", GEMM: "GEMM"}
JOBS = {CONV3: 9, UPCONV: 16, CONV4S2: 16, GEMM: 1}
KH_S2 = ((1, 3), (2, 0))            # CONV4S2 dgrad parity taps (tools/probe_conv.py)
EPI_ADD, EPI_LRELU_MASK = 1, 2
ACT_LRELU = 2

U_BF16 = 2.0 ** -8
U_ACC = 2.0 ** -23
U32 = 2.0 ** -24
LAMBDA = 10.0
TINY = 1e-30


def gamma(n, u=U_ACC):
    """Probabilistic bound factor of a chain of n roundings of unit roundoff u (see the module docstring)."""
    return math.expm1(LAMBDA * math.sqrt(n) * u + n * u * u / (1.0 - u))


def _planes(t, split):
    """Operand as float64; split: a (3, ...) bf16 pack of the fp32-accurate mode, summed back to its fp32 value."""
    return t.double().sum(0) if split else t.double()


# ------------------------------------------------------------------------------------------------ layouts
def out_hw(kind, H, W):
    if kind == UPCONV:
        return 2 * H, 2 * W
    if kind == CONV4S2:
        return H // 2, W // 2
    return H, W


def wpk_from_wpkT(kind, wT, Cout, Cin):
    """dgrad operand -> fprop operand layout (inverse of the per-kind transpose of the packing)."""
    if kind == GEMM:
        return wT.reshape(Cin, Cout).t()
    if kind == CONV3:
        return wT.reshape(Cin, 9, Cout).permute(2, 1, 0)
    if kind == UPCONV:
        return wT.reshape(Cin, 4, 4, Cout).permute(1, 3, 2, 0)
    wT = wT.reshape(4, Cin, 4, Cout)
    w = wT.new_zeros(Cout, 16, Cin)
    for py in range(2):
        for px in range(2):
            for a in range(2):
                for b in range(2):
                    w[:, KH_S2[py][a] * 4 + KH_S2[px][b], :] = wT[py * 2 + px, :, a * 2 + b, :].t()
    return w


def dwpk_from_wpk_grad(kind, g, Cout, Cin):
    """gradient in the wpk layout -> the (Cout, JOBS, Cin) wgrad accumulator layout."""
    if kind == UPCONV:
        return g.permute(1, 0, 2, 3).reshape(Cout, 16, Cin)
    return g.reshape(Cout, JOBS[kind], Cin)


def _wpk_view(kind, w, Cout, Cin):
    if kind == UPCONV:
        return w.reshape(4, Cout, 4, Cin)
    if kind == GEMM:
        return w.reshape(Cout, Cin)
    return w.reshape(Cout, JOBS[kind], Cin)


# ------------------------------------------------------------------------------------------------ references
def conv_ref(kind, x, w):
    """x (B,H,W,Cin) float64, w the fprop operand (wpk layout, float64) -> y (B,Ho,Wo,Cout): per-tap GEMMs."""
    B, H, W, Cin = x.shape
    if kind == GEMM:
        return x @ w.t()
    xp = torch.nn.functional.pad(x, (0, 0, 1, 1, 1, 1))
    if kind == CONV3:
        y = None
        for kh in range(3):
            for kw in range(3):
                t = xp[:, kh:kh + H, kw:kw + W, :] @ w[:, kh * 3 + kw, :].t()
                y = t if y is None else y + t
        return y
    if kind == CONV4S2:
        Ho, Wo = H // 2, W // 2
        y = None
        for kh in range(4):
            for kw in range(4):
                t = xp[:, kh:kh + 2 * Ho:2, kw:kw + 2 * Wo:2, :] @ w[:, kh * 4 + kw, :].t()
                y = t if y is None else y + t
        return y
    # UPCONV: output (2i+py, 2j+px), tap (a, b) reads input (i+py+a-1, j+px+b-1) with parity weights w[py*2+px]
    par = []
    for py in range(2):
        for px in range(2):
            acc = None
            for a in range(2):
                for b in range(2):
                    t = xp[:, py + a:py + a + H, px + b:px + b + W, :] @ w[py * 2 + px, :, a * 2 + b, :].t()
                    acc = t if acc is None else acc + t
            par.append(acc)
    Cout = par[0].shape[-1]
    y = torch.stack(par, 0).reshape(2, 2, B, H, W, Cout)
    return y.permute(2, 3, 0, 4, 1, 5).reshape(B, 2 * H, 2 * W, Cout)


def conv2d_ref(x, w, stride, ph, pw):
    """General kh x kw zero-padded conv (Inception): x (B,H,W,Cin), w (Cout,kh,kw,Cin) float64."""
    B, H, W, Cin = x.shape
    Cout, kh, kw, _ = w.shape
    Ho, Wo = (H + 2 * ph - kh) // stride + 1, (W + 2 * pw - kw) // stride + 1
    xp = torch.nn.functional.pad(x, (0, 0, pw, pw, ph, ph))
    y = None
    for i in range(kh):
        for j in range(kw):
            t = xp[:, i:i + stride * (Ho - 1) + 1:stride, j:j + stride * (Wo - 1) + 1:stride, :] @ w[:, i, j, :].t()
            y = t if y is None else y + t
    return y


def fprop_ref(kind, x, w):
    """-> (r, m) float64."""
    return conv_ref(kind, x, w), conv_ref(kind, x.abs(), w.abs())


def dgrad_ref(kind, dy, w, x_shape):
    """dy (B,Ho,Wo,Cout), w in the wpk layout -> (r, m) of dx (x_shape): VJPs of conv_ref."""
    out = []
    for d, ww in ((dy, w), (dy.abs(), w.abs())):
        x = torch.zeros(x_shape, dtype=torch.float64, device=dy.device, requires_grad=True)
        with torch.enable_grad():
            y = conv_ref(kind, x, ww)
            out.append(torch.autograd.grad(y, x, d)[0])
    return out[0], out[1]


def wgrad_ref(kind, x, dy, w_shape):
    """-> (r, m) of the weight gradient in the wpk layout (w_shape)."""
    out = []
    for xx, d in ((x, dy), (x.abs(), dy.abs())):
        w = torch.zeros(w_shape, dtype=torch.float64, device=x.device, requires_grad=True)
        with torch.enable_grad():
            y = conv_ref(kind, xx, w)
            out.append(torch.autograd.grad(y, w, d)[0])
    return out[0], out[1]


# ------------------------------------------------------------------------------------------------ bounds
def k_fprop(kind, Cin):
    return {CONV3: 9, UPCONV: 4, CONV4S2: 16, GEMM: 1}[kind] * Cin


def k_dgrad(kind, Cout):
    return {CONV3: 9, UPCONV: 16, CONV4S2: 4, GEMM: 1}[kind] * Cout


def k_wgrad(kind, B, H, W):
    return B * H * W // (4 if kind == CONV4S2 else 1)


def steps(K, splits=1):
    return -(-K // 16) + splits + 2


def ratio(got, r, bound):
    """max |got - r| / bound (inf if got has a non-finite element)."""
    got = got.double()
    if not bool(torch.isfinite(got).all()):
        return float("inf")
    return float(((got - r).abs() / (bound + TINY)).max()) if r.numel() else 0.0


def bound_bf16(r_out, e):
    """bf16-rounded output of a value within e of the float64 result; r_out the reference after the activation."""
    return U_BF16 * r_out.abs() + (1 + U_BF16) * e


def lrelu(t):
    return torch.where(t > 0, t, 0.2 * t)


def check_fprop(kind, x, wpk, got, Cout, splits=1, act=0, bias9=None, f32=False):
    """Worst |got - r| / bound of one fprop launch. x as given to the kernel (bf16, or fp32 in the fp32-accurate mode,
    whose wpk is the (3, ...) bf16 split)."""
    B, H, W, Cin = x.shape
    w = _wpk_view(kind, _planes(wpk, f32), Cout, Cin)
    r, m = fprop_ref(kind, x.double(), w)
    if bias9 is not None:
        bias = bias_from_bias9(bias9.double(), r.shape[1], r.shape[2])
        r, m = r + bias, m + bias.abs()
    n = steps(k_fprop(kind, Cin), splits)
    if f32:
        e = (2.0 ** -22 + gamma(n + 6)) * m
        if act == ACT_LRELU:
            r = lrelu(r)
        return ratio(got, r, e + U32 * r.abs())
    e = gamma(n) * m
    if act == ACT_LRELU:
        r = lrelu(r)
        e = e + U32 * r.abs()          # the fp32 product 0.2 * acc
    return ratio(got, r, bound_bf16(r, e))


def bias_from_bias9(bias9, H, W):
    """bias9 (B, 9, C) -> per-pixel bias (B, H, W, C): row ry*3+rx for ry in {top, interior, bottom}, rx likewise."""
    B, _, C = bias9.shape
    ry = torch.ones(H, dtype=torch.long, device=bias9.device)
    ry[0], ry[-1] = 0, 2
    rx = torch.ones(W, dtype=torch.long, device=bias9.device)
    rx[0], rx[-1] = 0, 2
    if H == 1:
        raise ValueError("bias9 border classes need H, W >= 2")
    cls = (ry[:, None] * 3 + rx[None, :]).reshape(-1)
    return bias9[:, cls, :].reshape(B, H, W, C)


def check_dgrad(kind, dy, wpkT, got, x_shape, splits=1, epi=None, f32=False):
    B, H, W, Cin = x_shape
    Cout = dy.shape[-1]
    w = wpk_from_wpkT(kind, _planes(wpkT, f32), Cout, Cin)
    r, m = dgrad_ref(kind, dy.double().reshape(B, *out_hw(kind, H, W), Cout), w, tuple(x_shape))
    n = steps(k_dgrad(kind, Cout), splits)
    e = ((2.0 ** -22 + gamma(n + 6)) if f32 else gamma(n)) * m
    q = r
    scale = 1.0
    if epi is not None:
        src, mode = epi[0].double().reshape(r.shape), epi[1]
        if mode == EPI_ADD:
            r = r + src
        else:
            scale = torch.where(src > 0, torch.ones_like(src), torch.full_like(src, 0.2))
            r = r * scale
    if f32:
        return ratio(got.reshape(r.shape), r, e * scale + 2 * U32 * (r.abs() + q.abs()))
    if epi is not None:
        e = (1 + U_BF16) * (e + U_BF16 * (q.abs() + e)) * scale
    return ratio(got.reshape(r.shape), r, bound_bf16(r, e))


def check_wgrad(kind, x, dy, got, old=None, slabs=1, f32=False):
    """got: the (Cout, JOBS, Cin) accumulator after the call; old: its value before (None: the call writes it)."""
    B, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    Ho, Wo = out_hw(kind, H, W)
    w_shape = (4, Cout, 4, Cin) if kind == UPCONV else ((Cout, Cin) if kind == GEMM else (Cout, JOBS[kind], Cin))
    r, m = wgrad_ref(kind, x.double(), dy.double().reshape(B, Ho, Wo, Cout), w_shape)
    r, m = dwpk_from_wpk_grad(kind, r, Cout, Cin), dwpk_from_wpk_grad(kind, m, Cout, Cin)
    if old is not None:
        r, m = r + old.double().reshape(r.shape), m + old.double().abs().reshape(r.shape)
    n = steps(k_wgrad(kind, B, H, W), slabs)
    e = ((2.0 ** -22 + gamma(n + 6)) if f32 else gamma(n)) * m
    return ratio(got.reshape(r.shape), r, e)


def check_stats(y, delta, groups):
    """delta: fp64 [groups][2][C], the change of the statistics slot across the call; y the tensor the call returned."""
    C = y.shape[-1]
    yy = y.double().reshape(groups, -1, C)
    rows = yy.shape[1]
    u = 2.0 ** -52 if y.dtype == torch.float32 else U32
    g = gamma(rows, u)
    d = delta.reshape(groups, 2, C)
    r1 = ratio(d[:, 0], yy.sum(1), g * yy.abs().sum(1) + 2.0 ** -50 * yy.abs().sum(1))
    r2 = ratio(d[:, 1], (yy * yy).sum(1), g * (yy * yy).sum(1) + 2.0 ** -50 * (yy * yy).sum(1))
    return max(r1, r2)


def check_conv2d(x, Cin, wpk, bias, got, kh, kw, stride, ph, pw, relu, x_c0):
    xs = x[..., x_c0:x_c0 + Cin].double()
    Cout = got.shape[-1]
    w = wpk.double().reshape(Cout, kh, kw, Cin)
    r, m = conv2d_ref(xs, w, stride, ph, pw), conv2d_ref(xs.abs(), w.abs(), stride, ph, pw)
    if bias is not None:
        r, m = r + bias.double(), m + bias.double().abs()
    if relu:
        r = r.clamp_min(0)
    return ratio(got, r, bound_bf16(r, gamma(steps(kh * kw * Cin)) * m))


def _cat(x1, x2):
    return x1.double() if x2 is None else torch.cat([x1.double(), x2.double()], 1)


def check_linear_fwd(x1, x2, w, bias, got):
    x = _cat(x1, x2)
    K = x.shape[1]
    wd = w.double()[:, :K]
    r, m = x @ wd.t(), x.abs() @ wd.abs().t()
    if bias is not None:
        r, m = r + bias.double(), m + bias.double().abs()
    e = gamma(K + 64) * m
    if got.dtype == torch.bfloat16:
        return ratio(got, r, bound_bf16(r, e))
    return ratio(got, r, e)


def check_linear_bwd_w(dy, x1, x2, dw, db, dw_old, db_old):
    x, d = _cat(x1, x2), dy.double()
    M = x.shape[0]
    r, m = d.t() @ x, d.abs().t() @ x.abs()
    rb, mb = d.sum(0), d.abs().sum(0)
    if dw_old is not None:
        r, m = r + dw_old.double().reshape(r.shape), m + dw_old.double().abs().reshape(r.shape)
    if db_old is not None:
        rb, mb = rb + db_old.double(), mb + db_old.double().abs()
    g = gamma(M + 64)
    out = ratio(dw.reshape(r.shape), r, g * m)
    if db is not None:
        out = max(out, ratio(db, rb, g * mb))
    return out


def check_linear_bwd_x(dy, w, got):
    d = dy.double()
    wd = w.double()[:, :got.shape[1]]
    r, m = d @ wd, d.abs() @ wd.abs()
    return ratio(got, r, gamma(d.shape[1] + 64) * m)


# ------------------------------------------------------------------------------------------------ call-time checker
class LaunchChecker:
    """Swaps the contraction entry points of sg2b200.ops for wrappers that synchronise the device, snapshot what the
    call accumulates into, run the original, synchronise, and check the result per element against float64 computed
    from the operands as they are at that moment. One row per (outermost) call in `rows`.

    keep(row) -> bool: the operands and output of that call are kept in `kept` (for fault-injection tests)."""

    NAMES = ("conv_fprop", "conv_dgrad", "conv_wgrad", "linear_fwd", "linear_bwd_w", "linear_bwd_x", "conv2d_fprop")
    # C entries of the contraction kernels: each one launched outside a wrapped call lands in `unchecked`
    ENTRIES = ("sg2_conv_fprop", "sg2_conv_dgrad", "sg2_conv_wgrad", "sg2_conv2d_fprop", "sg2_linear_fwd",
               "sg2_linear_bwd_w", "sg2_linear_bwd_x")

    def __init__(self, keep=None):
        from sg2b200 import ops
        self.ops = ops
        self.rows = []
        self.kept = []
        self.keep = keep
        self._depth = 0
        self._orig = {}
        self._launched = []
        self.calls = 0            # outermost wrapped calls made
        self.unchecked = []       # contraction entries launched outside a wrapped call

    def __enter__(self):
        ops = self.ops
        for n in self.NAMES:
            self._orig[n] = getattr(ops, n)
            setattr(ops, n, getattr(self, "_w_" + n))
        self._orig["_call"] = ops._call
        ops._call = self._rec_call
        return self

    def __exit__(self, *exc):
        for n, f in self._orig.items():
            setattr(self.ops, n, f)
        return False

    # every C entry called while a wrapped call runs (to read the split factor it resolved)
    def _rec_call(self, name, n_launch, *args):
        if self._depth:
            self._launched.append((name, args))
        elif name in self.ENTRIES:
            self.unchecked.append(name)
        return self._orig["_call"](name, n_launch, *args)

    def _run(self, name, *a, **kw):
        torch.cuda.synchronize()
        self._launched = []
        self.calls += 1
        self._depth += 1
        try:
            res = self._orig[name](*a, **kw)
        finally:
            self._depth -= 1
        torch.cuda.synchronize()
        return res

    def _splits(self, entry, idx):
        s = [args[idx] for n, args in self._launched if n == entry]
        return max(s) if s else 1

    def _row(self, row, worst, kept=None):
        row["ratio"] = worst
        self.rows.append(row)
        if kept is not None and self.keep is not None and self.keep(row):
            self.kept.append((row, kept))

    # ---- convolutions
    def _w_conv_fprop(self, kind, x, wpk, Cout, splitk=None, flop_scale=1.0, stats=None, groups=1, act=0, bias9=None):
        if self._depth:
            return self._orig["conv_fprop"](kind, x, wpk, Cout, splitk, flop_scale, stats, groups, act, bias9)
        st0 = stats.clone() if stats is not None else None
        res = self._run("conv_fprop", kind, x, wpk, Cout, splitk, flop_scale, stats, groups, act, bias9)
        y = res[0] if stats is not None else res
        f32 = x.dtype == torch.float32
        sp = self._splits("sg2_conv_fprop", 10) if not f32 else 1
        worst = check_fprop(kind, x, wpk, y, Cout, sp, act, bias9, f32)
        B, H, W, Cin = x.shape
        row = dict(op="fprop", kind=KIND_NAMES[kind], B=B, H=H, W=W, Cin=Cin, Cout=Cout, splitk=sp, groups=groups,
                   epi=("lrelu " if act == ACT_LRELU else "") + ("bias9 " if bias9 is not None else "") +
                   ("stats" if stats is not None else ""), dtype=str(x.dtype).split(".")[-1])
        if stats is not None:
            row["stats_ratio"] = check_stats(y, stats.double() - st0.double(), groups)
            worst = max(worst, row["stats_ratio"])
        self._row(row, worst, dict(x=x.clone(), wpk=wpk.clone(), y=y.clone(), splits=sp, act=act,
                                   bias9=None if bias9 is None else bias9.clone(), groups=groups,
                                   stats_delta=None if stats is None else (stats.double() - st0.double())))
        return res

    def _w_conv_dgrad(self, kind, dy, wpkT, B, H, W, Cin, splitk=None, flop_scale=1.0, epi=None):
        if self._depth:
            return self._orig["conv_dgrad"](kind, dy, wpkT, B, H, W, Cin, splitk, flop_scale, epi)
        epi_c = None if epi is None else (epi[0].clone(), epi[1])
        dx = self._run("conv_dgrad", kind, dy, wpkT, B, H, W, Cin, splitk, flop_scale, epi)
        f32 = dy.dtype == torch.float32
        sp = self._splits("sg2_conv_dgrad", 10) if not f32 else 1
        worst = check_dgrad(kind, dy, wpkT, dx, (B, H, W, Cin), sp, epi_c, f32)
        row = dict(op="dgrad", kind=KIND_NAMES[kind], B=B, H=H, W=W, Cin=Cin, Cout=dy.shape[-1], splitk=sp, groups=1,
                   epi={None: "", EPI_ADD: "add", EPI_LRELU_MASK: "lrelu_mask"}[None if epi is None else epi[1]],
                   dtype=str(dy.dtype).split(".")[-1])
        self._row(row, worst, dict(dy=dy.clone(), wpkT=wpkT.clone(), dx=dx.clone(), splits=sp, epi=epi_c))
        return dx

    def _w_conv_wgrad(self, kind, x, dy, dwpk, splitk=None, flop_scale=1.0, first=False):
        if self._depth:
            return self._orig["conv_wgrad"](kind, x, dy, dwpk, splitk, flop_scale, first)
        old = None if first else dwpk.clone()
        self._run("conv_wgrad", kind, x, dy, dwpk, splitk, flop_scale, first)
        f32 = x.dtype == torch.float32
        B, H, W, Cin = x.shape
        Cout = dy.shape[-1]
        calls = [args for n, args in self._launched if n == "sg2_conv_wgrad"]
        sp = max(a[9] for a in calls)
        slabs = 1
        if calls and calls[0][10] is not None:
            slabs = max(1, self.ops._lib.lib().sg2_conv_wgrad_slabs(kind, B, H, W, Cin, Cout, sp))
        worst = check_wgrad(kind, x, dy, dwpk, old, max(slabs, sp), f32)
        row = dict(op="wgrad", kind=KIND_NAMES[kind], B=B, H=H, W=W, Cin=Cin, Cout=Cout, splitk=sp, groups=1,
                   epi="first" if first else "accumulate", dtype=str(x.dtype).split(".")[-1], slabs=slabs)
        self._row(row, worst, dict(x=x.clone(), dy=dy.clone(), dwpk=dwpk.clone(),
                                   old=None if old is None else old, slabs=max(slabs, sp)))

    def _w_conv2d_fprop(self, x, Cin, wpk, bias, out, Cout, kh, kw, stride=1, ph=0, pw=0, relu=True, x_c0=0, out_c0=0):
        before = out.clone()
        res = self._run("conv2d_fprop", x, Cin, wpk, bias, out, Cout, kh, kw, stride, ph, pw, relu, x_c0, out_c0)
        worst = check_conv2d(x, Cin, wpk, bias, out[..., out_c0:out_c0 + Cout], kh, kw, stride, ph, pw, relu, x_c0)
        outside = torch.cat([out[..., :out_c0].reshape(-1), out[..., out_c0 + Cout:].reshape(-1)])
        inside_before = torch.cat([before[..., :out_c0].reshape(-1), before[..., out_c0 + Cout:].reshape(-1)])
        if not torch.equal(outside.view(torch.int16), inside_before.view(torch.int16)):
            worst = float("inf")                     # a byte outside the channel slice changed
        B, H, W, _ = x.shape
        self._row(dict(op="conv2d", kind=f"{kh}x{kw}s{stride}", B=B, H=H, W=W, Cin=Cin, Cout=Cout, splitk=1,
                       groups=1, epi="bias relu" if relu else "bias", dtype="bfloat16"), worst)
        return res

    # ---- linears
    def _w_linear_fwd(self, x1, x2, w, bias, out_bf16):
        out = self._run("linear_fwd", x1, x2, w, bias, out_bf16)
        self._row(dict(op="linear_fwd", kind="fc", B=x1.shape[0], H=1, W=1, Cin=x1.shape[1] + (0 if x2 is None else
                  x2.shape[1]), Cout=w.shape[0], splitk=1, groups=1, epi="bf16" if out_bf16 else "",
                       dtype="float32"), check_linear_fwd(x1, x2, w, bias, out))
        return out

    def _w_linear_bwd_w(self, dy, x1, x2, dw, db, accumulate=False):
        dw0 = dw.clone() if accumulate else None
        db0 = db.clone() if (accumulate and db is not None) else None
        self._run("linear_bwd_w", dy, x1, x2, dw, db, accumulate)
        self._row(dict(op="linear_bwd_w", kind="fc", B=x1.shape[0], H=1, W=1, Cin=x1.shape[1] + (0 if x2 is None else
                  x2.shape[1]), Cout=dy.shape[1], splitk=1, groups=1, epi="accumulate" if accumulate else "",
                       dtype=str(dy.dtype).split(".")[-1]), check_linear_bwd_w(dy, x1, x2, dw, db, dw0, db0))

    def _w_linear_bwd_x(self, dy, w, Kout):
        dx = self._run("linear_bwd_x", dy, w, Kout)
        self._row(dict(op="linear_bwd_x", kind="fc", B=dy.shape[0], H=1, W=1, Cin=Kout, Cout=dy.shape[1], splitk=1,
                       groups=1, epi="", dtype=str(dy.dtype).split(".")[-1]), check_linear_bwd_x(dy, w, dx))
        return dx

    # ---- report
    def worst_by_kind(self):
        out = {}
        for r in self.rows:
            k = f"{r['op']}/{r['kind']}/{r['dtype']}"
            out[k] = max(out.get(k, 0.0), r["ratio"])
        return out

    def table(self):
        cols = ("op", "kind", "B", "H", "W", "Cin", "Cout", "splitk", "groups", "epi", "ratio")
        lines = [" ".join(f"{c:>10}" for c in cols)]
        for r in self.rows:
            lines.append(" ".join(f"{r[c]:>10.3e}" if c == "ratio" else f"{str(r[c]):>10}" for c in cols))
        return "\n".join(lines)


def record(name, value, fname="step_launch_parity.json"):
    """Write a measured value to $SG2_RECORD_DIR/<fname> when that variable names a directory."""
    out = os.environ.get("SG2_RECORD_DIR")
    if not out or not os.path.isdir(out):
        return
    path = os.path.join(out, fname)
    d = json.load(open(path)) if os.path.exists(path) else {}
    d[name] = value
    json.dump(d, open(path, "w"), indent=1)


@contextmanager
def checked(keep=None):
    with LaunchChecker(keep) as c:
        yield c
