"""Tensor-level wrappers over the C ABI (include/sg2b200.h). Torch is plumbing only: it owns the memory and the
stream; every kernel launched here is one of ours. No CPU path: CPU tensors are rejected.

Layout convention: activations are NHWC bf16 torch tensors of shape (B, H, W, C) (or (P, C)).
"""
import ctypes
import os

import torch

from . import _lib

CONV3, UPCONV, CONV4S2, GEMM, STEM = 0, 1, 2, 3, 4
ACT_NONE, ACT_GLU, ACT_LRELU = 0, 1, 2
OUT_BF16, OUT_F32_ATOMIC, OUT_F32_STORE = 0, 1, 2
BN_EPS, BN_MOMENTUM = 1e-5, 0.1
N_SM = 148
# SMs a split-K launch is sized for: in the fused step several streams share the GPU, so a split layer does not have to
# fill every SM by itself — fewer splits = fewer fp32 slabs to write and re-read (SG2_SPLIT_SMS, measured in DESIGN.md)
SPLIT_SMS = int(os.environ.get("SG2_SPLIT_SMS", "148"))

_launches = 0   # kernels of ours launched through this module (bench.py reports it as gpu_launches)

# Reproducible reductions (default): split-K convolutions store per-split slabs that one pass sums in split order, weight
# gradients store per-split / per-CTA-lane slabs summed in order, every remaining cross-block sum (BatchNorm statistics,
# tap sums) is an fp64 atomic over per-block partials formed in a fixed order. SG2_DETERMINISTIC=0 switches the split-K
# and wgrad reductions back to fp32 red.global.add into a zeroed buffer (order not reproducible run to run).
DETERMINISTIC = os.environ.get("SG2_DETERMINISTIC", "1") != "0"
# Split-K reduction inside a thread-block cluster (the splits of a tile exchange their fp32 partial tiles through
# distributed shared memory and reduce them in rank order: no slab round trip, no finish launch). Largest cluster used
# (= cap of the split factor); 0 = always the slab path. Measured on the train step (ms/step): slabs 7.93, clusters of
# 2 / 3 / 4 / 6 / 8 / 16: 7.79 / 7.89 / 7.90 / 7.98 / 8.05 / 8.19 — a cluster is gang-scheduled onto free SMs of ONE GPC,
# which the other streams of the step make scarce, and in the shared GPU a split layer need not fill every SM itself.
CLUSTER_SPLITK = int(os.environ.get("SG2_CLUSTER_SPLITK", "2")) if DETERMINISTIC else 0


def launches():
    return _launches


_prof = None   # see profile_begin()


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("sg2b200 kernels need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("sg2b200: non-contiguous tensor passed to a kernel")
    if _prof is not None:
        _prof["keep"].append(t)      # recorded launches are replayed later: their operands must stay allocated
    return t.data_ptr()


def _p64(t):
    """Device pointer of an fp64 workspace (BatchNorm sums, tap sums)."""
    if t is not None and t.dtype != torch.float64:
        raise RuntimeError("sg2b200: this workspace is fp64 (torch.float64)")
    return _p(t)


def _call(name, n_launch, *args):
    global _launches
    _launches += n_launch
    _lib.call(name, *args)


# ---- optional recording of the convolution launches of a step (bench.py's roofline): every conv call made while
# recording is kept (entry point, raw arguments, executed FLOPs, operand tensors) so that the caller can replay exactly
# those launches, back to back in one CUDA graph, and time them with CUDA events without any host launch gaps.

def profile_begin():
    global _prof
    _prof = {"calls": [], "keep": []}


def profile_end():
    """-> (list of (name, args, flops), list of the tensors those calls reference)."""
    global _prof
    p, _prof = _prof, None
    return p["calls"], p["keep"]


def replay_call(name, args):
    """Re-issue a recorded conv call on the CURRENT stream (the stream is the last C argument)."""
    _lib.call(name, *(tuple(args[:-1]) + (_st(),)))


_TAPS_EFF = {0: 9, 1: 16, 2: 16, 3: 1}


def _conv_flops(kind, B, H, W, Cin, Cout):
    """MMA FLOPs one launch executes (fprop, dgrad and wgrad of a layer all contract the same index set)."""
    pix = B * (H // 2) * (W // 2) if kind == CONV4S2 else B * H * W
    return 2.0 * _TAPS_EFF[kind] * Cin * Cout * pix


def _conv_call(name, n_launch, flops, *args):
    _call(name, n_launch, *args)
    if _prof is not None:
        _prof["calls"].append((name, args, flops))


# ------------------------------------------------------------------------------------------ weights
JOBS = {CONV3: 9, UPCONV: 16, CONV4S2: 16, GEMM: 1, STEM: 1}


def pack_shapes(kind, CoP, CiP):
    if kind == CONV3:
        return (CoP, 9, CiP), (CiP, 9, CoP)
    if kind == UPCONV:
        return (4, CoP, 4, CiP), (CiP, 16, CoP)
    if kind == CONV4S2:
        return (CoP, 16, CiP), (4, CiP, 4, CoP)
    return (CoP, CiP), (CiP, CoP)


def pack_weights(kind, w, wpk, wpkT, Cout, Cin, CoP, CiP, ohwi=False):
    """fp32 master (OIHW, or [Cout][kh][kw][Cin] when ohwi) -> bf16 fprop / dgrad operand packs."""
    _call("sg2_pack_weights", 1, kind, _p(w), _p(wpk), _p(wpkT), Cout, Cin, CoP, CiP, int(ohwi), _st())


def pack_transpose(kind, wpk, wpkT, Cout, Cin):
    """dgrad operand from the bf16 fprop operand (per-tap [Cout][Cin] -> [Cin][Cout] transpose)."""
    _call("sg2_pack_transpose", 1, kind, _p(wpk), _p(wpkT), Cout, Cin, _st())


def unpack_wgrad(kind, dwpk, grad, Cout, Cin, CoP, CiP, accumulate, ohwi=False):
    _call("sg2_unpack_wgrad", 1, kind, _p(dwpk), _p(grad), Cout, Cin, CoP, CiP, int(accumulate), int(ohwi), _st())


# ------------------------------------------------------------------------------------------ convolutions
def _out_hw(kind, H, W):
    if kind == UPCONV:
        return 2 * H, 2 * W
    if kind == CONV4S2:
        return H // 2, W // 2
    return H, W


# gather kernels: two pixel tiles per CTA on the 256-channel instances (csrc/igemm.cuh FpropCfg; same switch as the C side)
IGEMM_MT2 = os.environ.get("SG2_IGEMM_MT2", "0") == "1"     # off: measured slower (conv.cu igemm_mt2)


def _gather_grid(Hg, Wg):
    """True when a conv with this per-group output grid runs on the gather kernel (conv.cu tile_eligible)."""
    return Hg < 16 or Wg < 8


def _auto_split(m_rows, n_cols, k_blocks, groups=1, cap=None, mt2=False):
    """Split-K factor for GEMMs whose 128 x BN output tiles cannot fill the 148 SMs.

    One CTA per (tile, split): the launch runs in ceil(tiles * s / 148) waves and a CTA's time is its K range plus a fixed
    part (prologue + epilogue; the fp32 red.global.add epilogue of a split CTA moves 4x the bytes of the bf16 store), both
    in units of one 64-deep K block. The factor with the smallest waves x (K / s + fixed) wins, the smaller one on ties —
    a factor that spills a few CTAs into a second wave costs a whole extra wave."""
    bn = n_cols if n_cols in (160, 192) else (
        256 if n_cols % 256 == 0 else (128 if n_cols % 128 == 0 else (64 if n_cols % 64 == 0 else 32)))
    m_tiles = -(-m_rows // 128)
    if mt2 and IGEMM_MT2 and bn == 256 and m_tiles >= 2:
        m_tiles = -(-m_tiles // 2)                    # units of two pixel tiles that share every weight stage
    tiles = m_tiles * max(1, n_cols // bn)
    if tiles >= 96 or k_blocks < 8:
        return 1
    if os.environ.get("SG2_SPLIT_OLD", "0") == "1":
        return max(1, min(k_blocks // 8, -(-N_SM // tiles)))
    tiles *= groups                                   # output-parity groups are separate GEMMs of the same launch
    best, best_cost = 1, None
    if cap is None:
        cap = CLUSTER_SPLITK if CLUSTER_SPLITK >= 2 else 32
    for sp in range(1, max(1, min(k_blocks // 8, cap)) + 1):     # >= 8 K blocks per CTA: little reduction work per output
        waves = -(-tiles * sp // SPLIT_SMS)
        cost = waves * (k_blocks / sp + (6.0 if sp > 1 else 3.0))
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = sp, cost
    return best


def _k_blocks(taps, ck):
    """K blocks of a launch: taps x (contraction channels / BK), BK as the kernels choose it."""
    bk = 64 if ck % 64 == 0 else (32 if ck % 32 == 0 else 16)
    return taps * max(1, ck // bk)


def conv_fprop(kind, x, wpk, Cout, splitk=None, flop_scale=1.0, stats=None, groups=1, act=ACT_NONE, bias9=None):
    """x (B,H,W,Cin) bf16 -> y bf16 (B,Ho,Wo,Cout).  (fp32 x + 3-plane packs: the fp32-accurate mode, see _conv3_f32.) With `stats` (fp32 [groups*2*Cout], zeroed) the per-channel sum /
    sum of squares of each of the `groups` sub-batches is accumulated too (in the conv epilogue, in the fp32->bf16 pass
    of a split-K layer, or by sg2_bn_stats when a pixel tile would straddle sub-batches); returns (y, True)."""
    if x.dtype == torch.float32:
        return _conv_fprop_f32(kind, x, wpk, Cout, stats, groups, act, bias9)
    B, H, W, Cin = x.shape
    fl = flop_scale * _conv_flops(kind, B, H, W, Cin, Cout)
    Ho, Wo = _out_hw(kind, H, W)
    taps = {CONV3: 9, UPCONV: 4, CONV4S2: 16, GEMM: 1}[kind]
    pgroups = 4 if kind == UPCONV else 1          # output parity groups (separate GEMMs)
    if splitk is None:
        gather = _gather_grid(*((H, W) if kind == UPCONV else (Ho, Wo))) and Cin % 64 == 0
        splitk = 1 if (act or bias9 is not None) else _auto_split(B * Ho * Wo // pgroups, Cout, taps * max(1, Cin // 64), pgroups,
                                                                  mt2=gather)
    splitk = max(1, min(splitk, _k_blocks(taps, Cin)))
    if 1 < splitk <= CLUSTER_SPLITK and Cin % 64 == 0 and Cout % 64 == 0:
        y = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=torch.bfloat16)
        try:
            _conv_call("sg2_conv_fprop", 1, fl, kind, _p(x), _p(wpk), _p(y), OUT_BF16, B, H, W, Cin, Cout, splitk,
                       _p64(stats), groups, act, None, _st())
            return y if stats is None else (y, True)
        except _lib.NoFuse:
            pass
    if splitk > 1:
        if DETERMINISTIC:
            y32 = torch.empty((splitk, B, Ho, Wo, Cout), device=x.device, dtype=torch.float32)
            _conv_call("sg2_conv_fprop", 2, fl, kind, _p(x), _p(wpk), _p(y32), OUT_F32_STORE, B, H, W, Cin, Cout, splitk,
                       None, 1, 0, None, _st())
            y = splitk_finish(y32, splitk, (B, Ho, Wo, Cout), stats, groups)
            return y if stats is None else (y, True)
        y32 = torch.zeros((B, Ho, Wo, Cout), device=x.device, dtype=torch.float32)
        _conv_call("sg2_conv_fprop", 2, fl, kind, _p(x), _p(wpk), _p(y32), OUT_F32_ATOMIC, B, H, W, Cin, Cout, splitk,
                   None, 1, 0, None, _st())
        if stats is None:
            return f32_to_bf16(y32)
        return f32_to_bf16_stats(y32, stats, groups), True
    y = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=torch.bfloat16)
    try:
        _conv_call("sg2_conv_fprop", 1, fl, kind, _p(x), _p(wpk), _p(y), OUT_BF16, B, H, W, Cin, Cout, 1, _p64(stats),
                   groups, act, _p(bias9), _st())
    except _lib.NoFuse:
        _conv_call("sg2_conv_fprop", 1, fl, kind, _p(x), _p(wpk), _p(y), OUT_BF16, B, H, W, Cin, Cout, 1, None, 1, act,
                   _p(bias9), _st())
        bn_stats(y.view(-1, Cout), stats, groups)
    return y if stats is None else (y, True)


EPI_ADD, EPI_LRELU_MASK = 1, 2


def _epi_apply(dx, epi):
    src, mode = epi
    return add_bf16(dx, src) if mode == EPI_ADD else lrelu_bwd(src, dx)


def conv_dgrad(kind, dy, wpkT, B, H, W, Cin, splitk=None, flop_scale=1.0, epi=None):
    """dy (B,Ho,Wo,Cout) bf16 -> dx bf16 (B,H,W,Cin). epi = (src, EPI_ADD | EPI_LRELU_MASK): src (shape of dx) is added
    to / masks the result, in the conv epilogue when the shape allows it, else by the separate kernel."""
    if dy.dtype == torch.float32:
        return _conv_dgrad_f32(kind, dy, wpkT, B, H, W, Cin, epi)
    Cout = dy.shape[-1]
    fl = flop_scale * _conv_flops(kind, B, H, W, Cin, Cout)
    taps = {CONV3: 9, UPCONV: 16, CONV4S2: 4, GEMM: 1}[kind]
    groups = 4 if kind == CONV4S2 else 1
    if splitk is None:
        gather = _gather_grid(*((H // 2, W // 2) if kind == CONV4S2 else (H, W))) and Cout % 64 == 0
        splitk = _auto_split(B * H * W // groups, Cin, taps * max(1, Cout // 64), groups, mt2=gather)
    splitk = max(1, min(splitk, _k_blocks(taps, Cout)))
    if 1 < splitk <= CLUSTER_SPLITK and Cin % 64 == 0 and Cout % 64 == 0:
        dx = torch.empty((B, H, W, Cin), device=dy.device, dtype=torch.bfloat16)
        try:
            _conv_call("sg2_conv_dgrad", 1, fl, kind, _p(dy), _p(wpkT), _p(dx), OUT_BF16, B, H, W, Cin, Cout, splitk,
                       _p(epi[0]) if epi is not None else None, epi[1] if epi is not None else 0, _st())
            return dx
        except _lib.NoFuse:
            pass
    if splitk > 1:
        if DETERMINISTIC:
            dx32 = torch.empty((splitk, B, H, W, Cin), device=dy.device, dtype=torch.float32)
            _conv_call("sg2_conv_dgrad", 2, fl, kind, _p(dy), _p(wpkT), _p(dx32), OUT_F32_STORE, B, H, W, Cin, Cout, splitk,
                       None, 0, _st())
            return splitk_finish(dx32, splitk, (B, H, W, Cin), None, 1, epi)      # + the epilogue operand, same pass
        dx32 = torch.zeros((B, H, W, Cin), device=dy.device, dtype=torch.float32)
        _conv_call("sg2_conv_dgrad", 2, fl, kind, _p(dy), _p(wpkT), _p(dx32), OUT_F32_ATOMIC, B, H, W, Cin, Cout, splitk,
                   None, 0, _st())
        dx = f32_to_bf16(dx32)
        return dx if epi is None else _epi_apply(dx, epi)
    dx = torch.empty((B, H, W, Cin), device=dy.device, dtype=torch.bfloat16)
    if epi is not None:
        try:
            _conv_call("sg2_conv_dgrad", 1, fl, kind, _p(dy), _p(wpkT), _p(dx), OUT_BF16, B, H, W, Cin, Cout, 1,
                       _p(epi[0]), epi[1], _st())
            return dx
        except _lib.NoFuse:
            pass
    _conv_call("sg2_conv_dgrad", 1, fl, kind, _p(dy), _p(wpkT), _p(dx), OUT_BF16, B, H, W, Cin, Cout, 1, None, 0, _st())
    return dx if epi is None else _epi_apply(dx, epi)


def conv_wgrad(kind, x, dy, dwpk, splitk=None, flop_scale=1.0, first=False):
    """dwpk (Cout, jobs, Cin) fp32 += dy^T im2col(x).  first: dwpk holds nothing yet (write instead of accumulate)."""
    if x.dtype == torch.float32:
        xs, dys = split3(x), split3(dy)
        for k, (i, j) in enumerate(_PAIRS):
            conv_wgrad(kind, xs[i], dys[j], dwpk, splitk, flop_scale, first and k == 0)
        return
    B, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    fl = flop_scale * _conv_flops(kind, B, H, W, Cin, Cout)
    if splitk is None:
        pix = dy.shape[0] * dy.shape[1] * dy.shape[2] // (4 if kind == UPCONV else 1)
        ktiles = max(1, pix // 64)
        bn = 16 if Cin <= 16 else (32 if Cin <= 32 else (64 if Cin <= 64 else (128 if Cin <= 128 else 256)))
        ctas = -(-Cout // 128) * -(-Cin // bn) * JOBS[kind]
        smax = ktiles // 2 if ktiles >= 2 else 1
        splitk = max(1, min(smax, -(-2 * N_SM // ctas)))
        if os.environ.get("SG2_WGRAD_WAVES", "0") == "1":
            # not measured yet (round 2 A/B): the wave accounting of _auto_split for the one-CTA-per-tap wgrad kernel
            best, best_cost = 1, None
            for sp in range(1, max(1, min(smax, 64)) + 1):
                cost = -(-ctas * sp // N_SM) * (ktiles / sp + 4.0)
                if best_cost is None or cost < best_cost - 1e-9:
                    best, best_cost = sp, cost
            splitk = best
    if not DETERMINISTIC:
        _conv_call("sg2_conv_wgrad", 1, fl, kind, _p(x), _p(dy), _p(dwpk), B, H, W, Cin, Cout, splitk, None, _st())
        return
    n = dwpk.numel()
    if splitk > 1 and n * 4 >= (16 << 20):
        splitk = max(1, min(splitk, (64 << 20) // (n * 4)))       # bound the slab traffic of large weights
    slabs = _lib.lib().sg2_conv_wgrad_slabs(kind, B, H, W, Cin, Cout, splitk)
    if slabs < 1:
        _lib.check(slabs if slabs < 0 else -1, "sg2_conv_wgrad_slabs")
    if slabs == 1 and first:
        # one slab and nothing to add to: the kernel stores straight into the accumulator
        _conv_call("sg2_conv_wgrad", 1, fl, kind, _p(x), _p(dy), _p(dwpk), B, H, W, Cin, Cout, splitk, _p(dwpk), _st())
        return
    parts = torch.empty((slabs, n), device=dwpk.device, dtype=torch.float32)
    _conv_call("sg2_conv_wgrad", 1, fl, kind, _p(x), _p(dy), _p(dwpk), B, H, W, Cin, Cout, splitk, _p(parts), _st())
    reduce_slabs(parts, slabs, n, dwpk, accumulate=not first)


def reduce_slabs(parts, nslabs, n, dst, accumulate):
    """dst (=|+=) the sum of the slabs, in slab order."""
    _call("sg2_reduce_slabs", 1, _p(parts), nslabs, n, n, _p(dst), int(accumulate), _st())


def splitk_finish(parts, nsplit, shape, stats=None, groups=1, epi=None):
    """(nsplit, *shape) fp32 split-K slabs -> bf16 tensor of `shape`: slabs summed in order (+ epilogue operand, + BN stats)."""
    C = shape[-1]
    y = torch.empty(shape, device=parts.device, dtype=torch.bfloat16)
    n = y.numel()
    _call("sg2_splitk_finish", 1, _p(parts), nsplit, n, _p(y), n // C, C, groups, _p64(stats),
          _p(epi[0]) if epi is not None else None, epi[1] if epi is not None else 0, _st())
    return y


# ------------------------------------------------------------------------------------------ fp32-accurate mode
# (hi,hi) ... (mid,mid) cross terms of the 3-way bf16 split, smallest first (see csrc/precise.cu and sg2b200.h)
_PAIRS = ((1, 1), (0, 2), (2, 0), (0, 1), (1, 0), (0, 0))


def split3(x):
    """fp32 tensor -> bf16 (3, *shape): x = hi + mid + lo to ~2^-24."""
    out = torch.empty((3,) + tuple(x.shape), device=x.device, dtype=torch.bfloat16)
    _call("sg2_split3", 1, _p(x), _p(out), x.numel(), _st())
    return out


def pack_weights_split3(kind, w, Cout, Cin, CoP, CiP, ohwi=False):
    """fp32 master -> (fprop packs, dgrad packs), each bf16 (3, *pack shape)."""
    s1, s2 = pack_shapes(GEMM if kind == STEM else kind, CoP, CiP)
    a = torch.empty(s1, device=w.device, dtype=torch.float32)
    b = torch.empty(s2, device=w.device, dtype=torch.float32)
    _call("sg2_pack_weights_f32", 1, kind, _p(w), _p(a), _p(b), Cout, Cin, CoP, CiP, int(ohwi), _st())
    return split3(a), split3(b)


def _conv_fprop_f32(kind, x, wpk3, Cout, stats, groups, act, bias9):
    B, H, W, Cin = x.shape
    Ho, Wo = _out_hw(kind, H, W)
    xs = split3(x)
    y = torch.zeros((B, Ho, Wo, Cout), device=x.device, dtype=torch.float32)
    for i, j in _PAIRS:
        _call("sg2_conv_fprop", 1, kind, _p(xs[i]), _p(wpk3[j]), _p(y), OUT_F32_ATOMIC, B, H, W, Cin, Cout, 1, None, 1, 0,
              None, _st())
    if bias9 is not None or act:
        _call("sg2_conv_post_f32", 1, _p(y), _p(bias9), act, B, Ho, Wo, Cout, _st())
    if stats is None:
        return y
    _call("sg2_bn_stats_f32", 1, _p(y), y.numel() // Cout, Cout, groups, _p64(stats), _st())
    return y, True


def _conv_dgrad_f32(kind, dy, wpkT3, B, H, W, Cin, epi):
    Cout = dy.shape[-1]
    dys = split3(dy)
    dx = torch.zeros((B, H, W, Cin), device=dy.device, dtype=torch.float32)
    for i, j in _PAIRS:
        _call("sg2_conv_dgrad", 1, kind, _p(dys[i]), _p(wpkT3[j]), _p(dx), OUT_F32_ATOMIC, B, H, W, Cin, Cout, 1, None, 0,
              _st())
    return dx if epi is None else _epi_apply(dx, epi)


# ------------------------------------------------------------------------------------------ BN / activations
class _ZeroArena:
    """Ring of zero-initialised scratch for the per-layer BatchNorm sums (fp32 forward, fp64 backward).

    A slot is handed out zeroed, accumulated into by one kernel and read by the next one on the same stream, then
    never touched again, so instead of one clearing launch per layer the arena clears half of itself whenever the
    bump pointer enters that half (everything that used it is already ordered before the clear on the stream)."""
    SIZE = 16 << 20

    def __init__(self, device):
        self.buf = torch.zeros(self.SIZE, device=device, dtype=torch.uint8)
        self.off = 0

    def take(self, nbytes, dtype):
        half = self.SIZE // 2
        n = -(-nbytes // 256) * 256
        if n > half:
            raise RuntimeError("sg2b200: BatchNorm scratch request too large")
        o = self.off % self.SIZE
        if (o % half) + n > half:              # do not straddle a half: move to the start of the next one
            o = (o // half + 1) * half % self.SIZE
        if o % half == 0 and not (o == 0 and self.off == 0):
            self.buf[o:o + half].zero_()       # entering a half: clear it (one fill per ~8 MB of slots)
        self.off = o + n
        return self.buf[o:o + nbytes].view(dtype)


_arenas = {}


def _arena(device):
    key = (device.index, torch.cuda.current_stream().cuda_stream)
    a = _arenas.get(key)
    if a is None:
        a = _arenas[key] = _ZeroArena(device)
    return a


def arena_reset(device):
    """Start of a train step: rewind and clear the scratch ring, so a CUDA-graph capture of the step contains every
    clear its slots need (a replay reuses the same slots each time)."""
    a = _arena(device)
    a.off = 0
    a.buf.zero_()


def bn_stats32(C, device, groups=1):
    """Zeroed fp64 [groups][2][C] slot for the per-channel sum / sum of squares (filled by a conv epilogue or bn_stats)."""
    return _arena(device).take(groups * 2 * C * 8, torch.float64)


def bn_stats(x2d, stats, groups=1):
    P, C = x2d.shape
    _call("sg2_bn_stats_f32" if x2d.dtype == torch.float32 else "sg2_bn_stats", 1, _p(x2d), P, C, groups, _p64(stats), _st())


def f32_to_bf16_stats(x32, stats, groups=1, keep_f32=False):
    """fp32 [..., C] -> bf16 copy, and += per-channel sums of the rounded values into `stats`.
    keep_f32 (fp32-accurate mode): no rounding — returns x32 itself with its exact statistics."""
    C = x32.shape[-1]
    if keep_f32:
        bn_stats(x32.view(-1, C), stats, groups)
        return x32
    y = torch.empty(x32.shape, device=x32.device, dtype=torch.bfloat16)
    _call("sg2_f32_to_bf16_stats", 1, _p(x32), _p(y), x32.numel() // C, C, groups, _p64(stats), _st())
    return y


def bn_eval_stats(rmean, rvar):
    C = rmean.numel()
    mean = torch.empty(C, device=rmean.device, dtype=torch.float32)
    rstd = torch.empty_like(mean)
    _call("sg2_bn_eval_prepare", 1, _p(rmean), _p(rvar), BN_EPS, _p(mean), _p(rstd), C, _st())
    return mean, rstd


def bn_act_fwd(x, gamma, beta, act, residual=None, stats=None, mean=None, rstd=None, running=None, groups=1):
    """out = act(bn(x)) (+ residual).
    train: stats (fp32 sums) given -> returns (out, mean, rstd) with mean/rstd derived in the kernel; `running` =
           (running_mean, running_var, num_batches_tracked) is updated like nn.BatchNorm does.
    eval : mean/rstd given.   no BN: gamma is None.
    groups > 1: the rows are `groups` equal sub-batches, each normalised on its own statistics (mean/rstd [groups][C])."""
    C = x.shape[-1]
    P = x.numel() // C
    f32 = x.dtype == torch.float32
    fn = "sg2_bn_act_fwd_f32" if f32 else "sg2_bn_act_fwd"
    out = torch.empty(x.shape[:-1] + ((C // 2) if act == ACT_GLU else C,), device=x.device, dtype=x.dtype)
    if gamma is None:
        _call(fn, 1, _p(x), None, None, None, None, None, _p(residual), _p(out), P, C, 1, act, BN_EPS,
              BN_MOMENTUM, None, None, None, _st())
        return out
    if stats is not None:
        mr = torch.empty(2, groups * C, device=x.device, dtype=torch.float32)
        mean, rstd = mr[0], mr[1]
    rm, rv, nbt = running if (running is not None and stats is not None) else (None, None, None)
    _call(fn, 1 + f32, _p(x), _p64(stats), _p(mean), _p(rstd), _p(gamma), _p(beta), _p(residual), _p(out), P, C,
          groups, act, BN_EPS, BN_MOMENTUM, _p(rm), _p(rv), _p(nbt), _st())
    return (out, mean, rstd) if stats is not None else out


def bn_act_bwd(x, dout, mean, rstd, gamma, beta, act, dgamma=None, dbeta=None, accumulate=False, groups=1):
    """-> dx (shape of x, bf16); dgamma/dbeta (fp32, = or +=) are written into the given tensors."""
    C = x.shape[-1]
    P = x.numel() // C
    dx = torch.empty_like(x)
    sums = _arena(x.device).take(groups * 2 * C * 8, torch.float64)
    _call("sg2_bn_act_bwd_f32" if x.dtype == torch.float32 else "sg2_bn_act_bwd", 2, _p(x), _p(dout), _p(mean), _p(rstd),
          _p(gamma), _p(beta), _p64(sums), _p(dx), _p(dgamma), _p(dbeta), int(accumulate), P, C, groups, act, _st())
    return dx


def lrelu_bwd(x, dout):
    dx = torch.empty_like(x)
    if x.dtype == torch.float32:
        _call("sg2_ew_f32", 1, 1, _p(x), _p(dout), _p(dx), x.numel(), _st())
    else:
        _call("sg2_lrelu_bwd", 1, _p(x), _p(dout), _p(dx), x.numel(), _st())
    return dx


def add_bf16(a, b, out=None):
    """out = a + b, elementwise, in the activations' storage type (bf16, or fp32 in the fp32-accurate mode)."""
    out = torch.empty_like(a) if out is None else out
    if a.dtype == torch.float32:
        _call("sg2_ew_f32", 1, 0, _p(a), _p(b), _p(out), a.numel(), _st())
    else:
        _call("sg2_add_bf16", 1, _p(a), _p(b), _p(out), a.numel(), _st())
    return out


def f32_to_bf16(x, out=None):
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    _call("sg2_f32_to_bf16", 1, _p(x), _p(out), x.numel(), _st())
    return out


# ------------------------------------------------------------------------------------------ concat / heads / stems
def concat_c(c, h):
    B, H, W, Ch = h.shape
    E = c.shape[1]
    out = torch.empty((B, H, W, E + Ch), device=h.device, dtype=h.dtype)
    _call("sg2_concat_c_f32" if h.dtype == torch.float32 else "sg2_concat_c", 1, _p(c), _p(h), _p(out), B, H * W, E, Ch, _st())
    return out


def concat_c_bwd(dcat, E, dc, want_dh=True):
    B, H, W, Ct = dcat.shape
    Ch = Ct - E
    dh = torch.empty((B, H, W, Ch), device=dcat.device, dtype=dcat.dtype) if want_dh else None
    _call("sg2_concat_c_bwd_f32" if dcat.dtype == torch.float32 else "sg2_concat_c_bwd", 1, _p(dcat), _p(dh), _p(dc), B,
          H * W, E, Ch, _st())
    return dh


# jointConv with the broadcast c_code folded into a per-sample border-class bias (see include/sg2b200.h).
# wst = (w fp32 master of the full weight, so, se, st): element (o, e, tap) at w.flat[o*so + e*se + tap*st].
def joint_bias(c, wst, Cout):
    w, so, se, st = wst
    B, E = c.shape
    bias9 = torch.empty((B, 9, Cout), device=c.device, dtype=torch.float32)
    _call("sg2_joint_bias", 1, _p(c), _p(w), so, se, st, _p(bias9), B, E, Cout, _st())
    return bias9


def joint_tap_sums(dy):
    B, H, W, Cout = dy.shape
    R = _arena(dy.device).take(B * 9 * Cout * 8, torch.float64)
    S = torch.empty((B, 9, Cout), device=dy.device, dtype=torch.float32)
    _call("sg2_joint_tap_sums", 2, _p(dy), _p64(R), _p(S), B, H, W, Cout, _st())
    return S


def joint_c_bwd(S, c, wst, dc=None, dw=None, dw_accumulate=False):
    w, so, se, st = wst
    B, E = c.shape
    _call("sg2_joint_c_bwd", (dc is not None) + (dw is not None), _p(S), _p(c), _p(w), so, se, st, _p(dc), _p(dw),
          int(dw_accumulate), B, E, S.shape[2], _st())


def head_tanh_fwd(y, B, H, W):
    img = torch.empty((B, 3, H, W), device=y.device, dtype=torch.float32)
    _call("sg2_head_tanh_fwd_f32" if y.dtype == torch.float32 else "sg2_head_tanh_fwd", 1, _p(y), _p(img), B, H * W,
          y.shape[-1], _st())
    return img


def head_tanh_bwd(dimg, img, CP, f32=False):
    B, _, H, W = img.shape
    dy = torch.empty((B, H, W, CP), device=img.device, dtype=torch.float32 if f32 else torch.bfloat16)
    _call("sg2_head_tanh_bwd_f32" if f32 else "sg2_head_tanh_bwd", 1, _p(dimg), _p(img), _p(dy), B, H * W, CP, _st())
    return dy


def stem_im2col(img, out=None, f32=False):
    """(B,3,S,S) fp32 -> im2col rows (1,1,B*(S/2)^2,64) bf16 of the 4x4 s2 stem; `out`: a contiguous slice to fill."""
    B, _, S, _ = img.shape
    rows = B * (S // 2) * (S // 2)
    if f32 or (out is not None and out.dtype == torch.float32):
        if out is None:
            out = torch.empty((1, 1, rows, 64), device=img.device, dtype=torch.float32)
        elif out.numel() != rows * 64 or not out.is_contiguous():
            raise RuntimeError("sg2b200: stem_im2col: bad output slice")
        _call("sg2_stem_im2col_f32", 1, _p(img), _p(out), B, S, _st())
        return out
    if out is None:
        out = torch.empty((1, 1, rows, 64), device=img.device, dtype=torch.bfloat16)
    elif out.numel() != rows * 64 or not out.is_contiguous() or out.dtype != torch.bfloat16:
        raise RuntimeError("sg2b200: stem_im2col: bad output slice")
    _call("sg2_stem_im2col", 1, _p(img), _p(out), B, S, _st())
    return out


def stem_col2im(dcol, B, S):
    dimg = torch.empty((B, 3, S, S), device=dcol.device, dtype=torch.float32)
    _call("sg2_stem_col2im_f32" if dcol.dtype == torch.float32 else "sg2_stem_col2im", 1, _p(dcol), _p(dimg), B, S, _st())
    return dimg


def nhwc_to_nchw_f32(x):
    B, H, W, C = x.shape
    out = torch.empty((B, C * H * W), device=x.device, dtype=torch.float32)
    if x.dtype == torch.float32:
        _call("sg2_hwc_chw_f32", 1, _p(x), _p(out), B, H * W, C, 1, _st())
    else:
        _call("sg2_nhwc_to_nchw_f32", 1, _p(x), _p(out), B, H * W, C, _st())
    return out


def nchw_f32_to_nhwc(x, B, H, W, C, f32=False):
    out = torch.empty((B, H, W, C), device=x.device, dtype=torch.float32 if f32 else torch.bfloat16)
    if f32:
        _call("sg2_hwc_chw_f32", 1, _p(x), _p(out), B, H * W, C, 0, _st())
    else:
        _call("sg2_nchw_f32_to_nhwc", 1, _p(x), _p(out), B, H * W, C, _st())
    return out


# ------------------------------------------------------------------------------------------ small fp32 ops
def linear_fwd(x1, x2, w, bias, out_bf16):
    M, K1 = x1.shape
    K2 = 0 if x2 is None else x2.shape[1]
    N = w.shape[0]
    out = torch.empty((M, N), device=w.device, dtype=torch.bfloat16 if out_bf16 else torch.float32)
    _call("sg2_linear_fwd", 1, _p(x1), K1, _p(x2), K2, _p(w), _p(bias), _p(out), int(out_bf16), M, N, _st())
    return out


def linear_bwd_w(dy, x1, x2, dw, db, accumulate=False):
    M, K1 = x1.shape
    K2 = 0 if x2 is None else x2.shape[1]
    N = dy.shape[1]
    _call("sg2_linear_bwd_w", 1, _p(dy), int(dy.dtype == torch.bfloat16), _p(x1), K1, _p(x2), K2, _p(dw), _p(db),
          M, N, int(accumulate), _st())


def linear_bwd_x(dy, w, Kout):
    M, N = dy.shape
    dx = torch.empty((M, Kout), device=dy.device, dtype=torch.float32)
    scratch = torch.empty(_lib.lib().sg2_linear_bwd_x_scratch_floats(N, Kout), device=dy.device, dtype=torch.float32)
    _call("sg2_linear_bwd_x", 2, _p(dy), int(dy.dtype == torch.bfloat16), _p(w), _p(dx), _p(scratch), M, N, w.shape[1],
          Kout, _st())
    return dx


def ca_glu_reparam_fwd(fc, eps):
    B, E4 = fc.shape
    E = E4 // 4
    mu = torch.empty((B, E), device=fc.device, dtype=torch.float32)
    logvar, c = torch.empty_like(mu), torch.empty_like(mu)
    _call("sg2_ca_glu_reparam_fwd", 1, _p(fc), _p(eps), _p(mu), _p(logvar), _p(c), B, E, _st())
    return mu, logvar, c


def ca_glu_reparam_bwd(fc, eps, dmu, dlogvar, dc):
    B, E4 = fc.shape
    dfc = torch.empty_like(fc)
    _call("sg2_ca_glu_reparam_bwd", 1, _p(fc), _p(eps), _p(dmu), _p(dlogvar), _p(dc), _p(dfc), B, E4 // 4, _st())
    return dfc


def chw_hwc(x, B, C, HW, to_hwc):
    out = torch.empty_like(x)
    if x.dtype == torch.float32:
        _call("sg2_hwc_chw_f32", 1, _p(x), _p(out), B, HW, C, int(not to_hwc), _st())
    else:
        _call("sg2_chw_hwc_bf16", 1, _p(x), _p(out), B, C, HW, int(to_hwc), _st())
    return out


def logits_fwd(x, w, bias, out=None):
    B, H, W, C = x.shape
    prob = torch.empty(B, device=x.device, dtype=torch.float32) if out is None else out
    _call("sg2_logits_fwd_f32" if x.dtype == torch.float32 else "sg2_logits_fwd", 1, _p(x), _p(w), _p(bias), _p(prob), B,
          H * W, C, _st())
    return prob


def logits_bwd(dprob, prob, x, w, dx, dx_accumulate, dw, dbias):
    B, H, W, C = x.shape
    if x.dtype == torch.float32:
        _call("sg2_logits_bwd_f32", 1, _p(dprob), _p(prob), _p(x), _p(w), _p(dx), int(dx_accumulate), _p(dw), _p(dbias), B,
              H * W, C, _st())
        return
    scratch = None
    if dw is not None:
        scratch = torch.empty(_lib.lib().sg2_logits_bwd_scratch_floats(B, H * W, C), device=x.device, dtype=torch.float32)
    _call("sg2_logits_bwd", 1 + (dw is not None), _p(dprob), _p(prob), _p(x), _p(w), _p(dx), int(dx_accumulate), _p(dw),
          _p(dbias), _p(scratch), B, H * W, C, _st())


# ------------------------------------------------------------------------------------------ Inception-v3 scorer
def _slice_ptr(t, c0):
    """Device pointer of channel c0 of the NHWC tensor t (its pixel stride stays t.shape[-1] channels)."""
    if t.dtype != torch.bfloat16:
        raise RuntimeError("sg2b200: Inception activations are bf16")
    return _p(t) + 2 * c0


def conv2d_out_hw(H, W, kh, kw, stride, ph, pw):
    return (H + 2 * ph - kh) // stride + 1, (W + 2 * pw - kw) // stride + 1


def conv2d_plan(B, H, W, Cin, Cout, kh, kw, stride=1, ph=0, pw=0):
    """The tiling sg2_conv2d_fprop uses for this shape: dict of issued / useful MMA rows and columns, BN, BK, tile."""
    out = (ctypes.c_longlong * 8)()
    _lib.call("sg2_conv2d_plan", B, H, W, Cin, Cout, kh, kw, stride, ph, pw, ctypes.addressof(out))
    keys = ("issued_rows", "useful_rows", "issued_cols", "bn", "bk", "tw", "th", "nb")
    return dict(zip(keys, (int(v) for v in out)))


def conv2d_fprop(x, Cin, wpk, bias, out, Cout, kh, kw, stride=1, ph=0, pw=0, relu=True, x_c0=0, out_c0=0):
    """out[..., out_c0:out_c0+Cout] = relu?(conv(x[..., x_c0:x_c0+Cin], wpk) + bias); x, out NHWC bf16 (B, H, W, C)."""
    B, H, W, _ = x.shape
    Ho, Wo = conv2d_out_hw(H, W, kh, kw, stride, ph, pw)
    if tuple(out.shape[:3]) != (B, Ho, Wo) or x_c0 + Cin > x.shape[3] or out_c0 + Cout > out.shape[3]:
        raise RuntimeError(f"sg2b200: conv2d_fprop: shapes {tuple(x.shape)} -> {tuple(out.shape)} "
                           f"({kh}x{kw} s{stride}, channels {x_c0}+{Cin} -> {out_c0}+{Cout})")
    flops = 2.0 * B * Ho * Wo * Cout * Cin * kh * kw
    _conv_call("sg2_conv2d_fprop", 1, flops, _slice_ptr(x, x_c0), x.shape[3], _p(wpk), _p(bias),
               _slice_ptr(out, out_c0), out.shape[3], B, H, W, Cin, Cout, kh, kw, stride, ph, pw, int(relu), _st())
    return out


def inception_stem(img):
    """(B,3,S,S) fp32 in [-1, 1] -> (B,149,149,32) bf16 im2col rows of Conv2d_1a_3x3 of the preprocessed 299^2 image."""
    B, _, S, _ = img.shape
    col = torch.empty((B, 149, 149, 32), device=img.device, dtype=torch.bfloat16)
    _call("sg2_inception_stem", 1, _p(img), _p(col), B, S, _st())
    return col


def maxpool3s2(x, out=None, out_c0=0):
    B, H, W, C = x.shape
    Ho, Wo = (H - 3) // 2 + 1, (W - 3) // 2 + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, C), device=x.device, dtype=torch.bfloat16)
    if tuple(out.shape[:3]) != (B, Ho, Wo) or out_c0 + C > out.shape[3]:
        raise RuntimeError("sg2b200: maxpool3s2: bad output")
    _call("sg2_maxpool3s2", 1, _p(x), _slice_ptr(out, out_c0), out.shape[3], B, H, W, C, _st())
    return out


def avgpool3s1(x):
    B, H, W, C = x.shape
    out = torch.empty_like(x)
    _call("sg2_avgpool3s1", 1, _p(x), _p(out), B, H, W, C, _st())
    return out


def global_avg(x, out=None):
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty((B, C), device=x.device, dtype=torch.float32)
    _call("sg2_global_avg", 1, _p(x), _p(out), B, H * W, C, _st())
    return out


def softmax_rows(x, out=None):
    M, N = x.shape
    if out is None:
        out = torch.empty_like(x)
    _call("sg2_softmax_rows", 1, _p(x), _p(out), M, N, _st())
    return out
