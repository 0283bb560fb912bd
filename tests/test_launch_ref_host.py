"""CPU checks of tests/launch_ref.py: every float64 reference equals torch's float64 conv2d / interpolate / autograd on
the unpacked master weight, and the per-element bound accepts the exact result rounded like a kernel rounds it while
rejecting each seeded fault at the step's largest contraction lengths."""
import pytest
import torch
import torch.nn.functional as F

from tests import launch_ref as L
from tools.probe_conv import pack_ref, ref_fwd, unpack_wgrad_ref

KINDS = [L.CONV3, L.UPCONV, L.CONV4S2, L.GEMM]
KSIZE = {L.CONV3: 3, L.UPCONV: 3, L.CONV4S2: 4, L.GEMM: 1}


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _close(a, b, tol=1e-12):
    return float((a - b).abs().max()) <= tol * (1 + float(b.abs().max()))


@pytest.mark.parametrize("kind", KINDS)
def test_references_match_torch_float64(kind):
    """fprop from wpk, dgrad from wpkT, wgrad into the (Cout, JOBS, Cin) accumulator, against F.conv2d (after a nearest
    2x upsample for UPCONV) and its autograd on the OIHW master."""
    g = torch.Generator().manual_seed(kind)
    B, H, W, Ci, Co = 2, 6, 8, 5, 7
    k = KSIZE[kind]
    x = torch.randn(B, Ci, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(Co, Ci, k, k, generator=g, dtype=torch.float64, requires_grad=True)
    y = ref_fwd(kind, x, w)
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    dx, dw = torch.autograd.grad(y, (x, w), dy)
    wpk, wpkT = pack_ref(kind, w.detach())
    r, m = L.fprop_ref(kind, _nhwc(x.detach()), L._wpk_view(kind, wpk, Co, Ci))
    assert _close(r, _nhwc(y.detach()))
    assert bool((m >= r.abs() - 1e-12).all())
    wback = L.wpk_from_wpkT(kind, wpkT, Co, Ci)
    assert _close(wback, L._wpk_view(kind, wpk, Co, Ci))
    rdx, mdx = L.dgrad_ref(kind, _nhwc(dy), wback, (B, H, W, Ci))
    assert _close(rdx, _nhwc(dx)) and bool((mdx >= rdx.abs() - 1e-12).all())
    wshape = L._wpk_view(kind, wpk, Co, Ci).shape
    rdw, _ = L.wgrad_ref(kind, _nhwc(x.detach()), _nhwc(dy), wshape)
    dwpk = L.dwpk_from_wpk_grad(kind, rdw, Co, Ci)
    # unpack_wgrad_ref sums the UPCONV parity taps into an fp32 buffer
    assert _close(unpack_wgrad_ref(kind, dwpk, Co, Ci).double(), dw, 1e-12 if kind != L.UPCONV else 1e-6)


def test_bias9_is_the_folded_constant_channels():
    """conv3x3(cat(c broadcast, h)) == conv(h) + bias9 expanded by border class (include/sg2b200.h, sg2_joint_bias)."""
    g = torch.Generator().manual_seed(3)
    B, E, Ch, Co, H, W = 2, 3, 4, 5, 5, 7
    c = torch.randn(B, E, generator=g, dtype=torch.float64)
    h = torch.randn(B, Ch, H, W, generator=g, dtype=torch.float64)
    w = torch.randn(Co, E + Ch, 3, 3, generator=g, dtype=torch.float64)
    truth = F.conv2d(torch.cat([c[:, :, None, None].expand(B, E, H, W), h], 1), w, padding=1)
    bias9 = torch.zeros(B, 9, Co, dtype=torch.float64)
    for ry in range(3):
        for rx in range(3):
            for kh in range(3):
                for kw in range(3):
                    if (ry == 0 and kh == 0) or (ry == 2 and kh == 2) or (rx == 0 and kw == 0) or (rx == 2 and kw == 2):
                        continue
                    bias9[:, ry * 3 + rx] += c @ w[:, :E, kh, kw].t()
    wpk, _ = pack_ref(L.CONV3, w[:, E:])
    r = L.conv_ref(L.CONV3, _nhwc(h), wpk) + L.bias_from_bias9(bias9, H, W)
    assert _close(r, _nhwc(truth))
    # and check_fprop takes the same path: the exact result rounded to bf16 is accepted
    got = r.to(torch.bfloat16)
    assert L.check_fprop(L.CONV3, _nhwc(h), wpk, got, Co, bias9=bias9) <= 1.0


@pytest.mark.parametrize("mode", [L.EPI_ADD, L.EPI_LRELU_MASK])
def test_dgrad_epilogue_modes(mode):
    g = torch.Generator().manual_seed(mode)
    B, H, W, Ci, Co = 2, 8, 8, 16, 32
    dy = torch.randn(B, H, W, Co, generator=g).bfloat16()
    wpkT = torch.randn(Ci, 9, Co, generator=g).bfloat16()
    src = torch.randn(B, H, W, Ci, generator=g).bfloat16()
    w = L.wpk_from_wpkT(L.CONV3, wpkT.double(), Co, Ci)
    q, _ = L.dgrad_ref(L.CONV3, dy.double(), w, (B, H, W, Ci))
    truth = q + src.double() if mode == L.EPI_ADD else q * torch.where(src.double() > 0, 1.0, 0.2)
    lr = F.leaky_relu(src.double(), 0.2)     # the mask is the LeakyReLU(0.2) derivative at src
    if mode == L.EPI_LRELU_MASK:
        assert _close(truth, q * torch.where(lr > 0, 1.0, 0.2))
    fused = truth.to(torch.bfloat16)
    separate = (q.to(torch.bfloat16).double() + src.double() if mode == L.EPI_ADD else
                q.to(torch.bfloat16).double() * torch.where(src.double() > 0, 1.0, 0.2)).to(torch.bfloat16)
    for got in (fused, separate):
        assert L.check_dgrad(L.CONV3, dy, wpkT, got, (B, H, W, Ci), epi=(src, mode)) <= 1.0
    assert L.check_dgrad(L.CONV3, dy, wpkT, q.to(torch.bfloat16), (B, H, W, Ci), epi=(src, mode)) > 1.0


# ----------------------------------------------------------------------------------------- sensitivity
def _big_fprop():
    """The step's largest fprop contraction: CONV3 over 2048 channels (K = 18 432), on 128 output pixels."""
    g = torch.Generator().manual_seed(7)
    B, H, W, Ci, Co = 8, 4, 4, 2048, 16
    x = torch.randn(B, H, W, Ci, generator=g).bfloat16()
    wpk = torch.randn(Co, 9, Ci, generator=g).bfloat16()
    r, _ = L.fprop_ref(L.CONV3, x.double(), wpk.double())
    return x, wpk, r, Co


def test_fprop_fault_sensitivity_at_k_18432():
    x, wpk, r, Co = _big_fprop()
    ok = r.to(torch.bfloat16)
    assert L.check_fprop(L.CONV3, x, wpk, ok, Co) <= 1.0
    xd, wd = x.double(), wpk.double()
    faults = {}
    # one border tap dropped for one output pixel: pixel (0, 1) of image 3, tap (kh, kw) = (2, 1) reads x[3, 1, 1]
    t = r.clone()
    t[3, 0, 1] -= xd[3, 1, 1] @ wd[:, 7, :].t()
    faults["border tap"] = t
    # one 16-channel K block (channels 512..527 of tap 4) dropped from the one 128-row pixel tile
    t = r.clone()
    t -= xd[..., 512:528] @ wd[:, 4, 512:528].t()
    faults["K block"] = t
    # one output row (pixel row 2 of image 5) taken from the neighbouring image
    t = r.clone()
    t[5, 2] = r[4, 2]
    faults["neighbour image"] = t
    # one untouched element left at a stale value (the previous launch's output at that position)
    g = torch.Generator().manual_seed(8)
    stale, _ = L.fprop_ref(L.CONV3, torch.randn(x.shape, generator=g).bfloat16().double(), wd)
    t = r.clone()
    t[6, 3, 3, 9] = stale[6, 3, 3, 9]
    faults["stale element"] = t
    for name, t in faults.items():
        assert L.check_fprop(L.CONV3, x, wpk, t.to(torch.bfloat16), Co) > 1.0, name


def test_dgrad_fault_sensitivity_at_k_18432():
    """dgrad of a 2048-output-channel CONV3: K = 9 x 2048 again; one tap of one border pixel dropped."""
    g = torch.Generator().manual_seed(9)
    B, H, W, Ci, Co = 2, 4, 4, 16, 2048
    dy = torch.randn(B, H, W, Co, generator=g).bfloat16()
    wpkT = torch.randn(Ci, 9, Co, generator=g).bfloat16()
    w = L.wpk_from_wpkT(L.CONV3, wpkT.double(), Co, Ci)
    r, _ = L.dgrad_ref(L.CONV3, dy.double(), w, (B, H, W, Ci))
    assert L.check_dgrad(L.CONV3, dy, wpkT, r.to(torch.bfloat16), (B, H, W, Ci)) <= 1.0
    t = r.clone()
    # dx[1, 0, 3] receives dy[1, 1, 2] through tap (kh, kw) = (2, 0) (dx[i] += dy[i - kh + 1] w[tap])
    t[1, 0, 3] -= dy[1, 1, 2].double() @ w[:, 6, :]
    assert L.check_dgrad(L.CONV3, dy, wpkT, t.to(torch.bfloat16), (B, H, W, Ci)) > 1.0
    t = r.clone()
    t[0, 1] = r[1, 1]
    assert L.check_dgrad(L.CONV3, dy, wpkT, t.to(torch.bfloat16), (B, H, W, Ci)) > 1.0


def test_stats_wrong_group_rejected():
    """72-row discriminator pass: 3 groups of 24 x 64^2 rows (the first statistics layer of D_NET256)."""
    g = torch.Generator().manual_seed(10)
    groups, rows, C = 3, 24 * 64 * 64, 16
    y = torch.randn(groups * rows, C, generator=g).bfloat16()
    yy = y.double().reshape(groups, rows, C)
    delta = torch.stack([yy.sum(1), (yy * yy).sum(1)], 1)           # [groups][2][C]
    assert L.check_stats(y, delta.float().double(), groups) <= 1.0   # fp32-rounded sums are within the bound
    bad = delta.clone()
    bad[1, :, 5] = delta[2, :, 5]
    assert L.check_stats(y, bad, groups) > 1.0


def _wgrad_case(P, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(1, 1, P, 16, generator=g).bfloat16()
    dy = torch.randn(1, 1, P, 16, generator=g).bfloat16()
    r, _ = L.wgrad_ref(L.GEMM, x.double(), dy.double(), (16, 16))
    return x, dy, r.reshape(16, 1, 16)


def _drop(x, dy, r, p0, npx):
    part = dy[0, 0, p0:p0 + npx].double().t() @ x[0, 0, p0:p0 + npx].double()
    return (r - part.reshape(r.shape)).float()


def test_wgrad_dropped_tile_at_8192_pixels():
    x, dy, r = _wgrad_case(8192, 11)
    assert L.check_wgrad(L.GEMM, x, dy, r.float()) <= 1.0
    assert L.check_wgrad(L.GEMM, x, dy, _drop(x, dy, r, 3 * 128, 128)) > 1.0
    # accumulate mode: the change across the call is what is checked
    old = torch.randn(r.shape, generator=torch.Generator().manual_seed(12)) * 50
    assert L.check_wgrad(L.GEMM, x, dy, (r + old.double()).float(), old=old) <= 1.0
    assert L.check_wgrad(L.GEMM, x, dy, (_drop(x, dy, r, 0, 128).double() + old.double()).float(), old=old) > 1.0


def test_wgrad_smallest_caught_fault_at_1_6m_pixels():
    """24 x 256^2 pixels: one dropped 128-pixel tile of zero-mean data is below the bound (module docstring); a dropped
    run of 256 tiles (2 % of the pixels) is the smallest fault the bound catches here."""
    P = 24 * 256 * 256
    x, dy, r = _wgrad_case(P, 13)
    assert L.check_wgrad(L.GEMM, x, dy, r.float()) <= 1.0
    assert L.check_wgrad(L.GEMM, x, dy, _drop(x, dy, r, 5000 * 128, 128)) <= 1.0
    assert L.check_wgrad(L.GEMM, x, dy, _drop(x, dy, r, 5000 * 128, 256 * 128)) > 1.0


def test_conv2d_and_linear_references():
    g = torch.Generator().manual_seed(14)
    x = torch.randn(2, 9, 9, 24, generator=g, dtype=torch.float64)
    w = torch.randn(8, 3, 5, 16, generator=g, dtype=torch.float64)
    b = torch.randn(8, generator=g, dtype=torch.float64)
    truth = F.relu(F.conv2d(x[..., 4:20].permute(0, 3, 1, 2), w.permute(0, 3, 1, 2), b, stride=2, padding=(1, 2)))
    got = _nhwc(truth).to(torch.bfloat16)
    assert L.check_conv2d(x, 16, w.reshape(8, -1), b, got, 3, 5, 2, 1, 2, True, 4) <= 1.0
    bad = got.clone()
    bad[1, 2, 3, 4] = got[1, 2, 2, 4] + 1
    assert L.check_conv2d(x, 16, w.reshape(8, -1), b, bad, 3, 5, 2, 1, 2, True, 4) > 1.0
    x1, x2 = torch.randn(6, 10, generator=g), torch.randn(6, 4, generator=g)
    wl, bl = torch.randn(12, 14, generator=g), torch.randn(12, generator=g)
    y = F.linear(torch.cat([x1, x2], 1).double(), wl.double(), bl.double())
    assert L.check_linear_fwd(x1, x2, wl, bl, y.float()) <= 1.0
    assert L.check_linear_fwd(x1, x2, wl, bl, y.to(torch.bfloat16)) <= 1.0
    y2 = y.clone()
    y2[3, 5] += 1e-3 * y.abs().max()
    assert L.check_linear_fwd(x1, x2, wl, bl, y2.float()) > 1.0
    dy = torch.randn(6, 12, generator=g)
    dw = (dy.double().t() @ torch.cat([x1, x2], 1).double()).float()
    assert L.check_linear_bwd_w(dy, x1, x2, dw, dy.double().sum(0).float(), None, None) <= 1.0
    assert L.check_linear_bwd_x(dy, wl, (dy.double() @ wl.double()[:, :10]).float()) <= 1.0
