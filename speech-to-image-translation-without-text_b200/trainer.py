"""Fused train step: the inner loop of the reference's condGANTrainer.train (StackGAN_v2/trainer.py:529-572, minus
the out-of-scope Inception scoring) scheduled by hand over the sg2b200 engines — no autograd graph, no Python-side
loss arithmetic.

    step = G forward -> for each D: train_Dnet (real / wrong / fake passes, 6 BCE terms, backward, Adam)
           -> train_Gnet (D forwards on the live fakes, BCE + class-aware + KL losses, backward through the Ds
              and G, Adam) -> EMA of the generator weights

Differences from the reference that do not change any result (SURVEY.md section 7, "wasted reference work"):
no dgrad into real/wrong images, no D weight gradients in the G step (the reference zeroes them before use,
trainer.py:385), the three D passes accumulate their weight gradients in one packed fp32 buffer.

Parameters, Adam moments, EMA shadow and gradients of each network live in flat fp32 buckets (one Adam launch per
network; the gradient bucket is what NCCL all-reduces in the data-parallel run).
"""
import ctypes
import os

import torch

from . import ops
from .nets import GradSink

_st = ops._st
_p = ops._p


def _is_ohwi(p):
    """Conv weights (except the Cout = 1 logit convs, which run as dot products) are stored [Cout][kh][kw][Cin]."""
    return p.dim() == 4 and p.shape[0] > 1


class FlatBucket:
    """All parameters of one network as views of a single flat fp32 buffer (+ grad / Adam m, v / optional EMA).

    Conv weights are STORED in the layout the kernels consume, [Cout][kh][kw][Cin] ("OHWI"), and exposed to torch as
    OIHW-shaped strided views (`p.data`), so state_dict / load_state_dict / checkpoints keep the reference's shapes.
    Adam, EMA and the NCCL all-reduce are elementwise over the flat buffers and do not care about the layout; what it
    buys: the bf16 fprop operand of a CONV3x3 / CONV4x4S2 layer is a plain cast of the master (the Adam kernel writes
    it as a bf16 mirror of the bucket) and the wgrad kernels accumulate straight into the gradient bucket."""

    # elements: conv weights at least this large are all-reduced one by one as soon as their wgrad is done (data-parallel
    # runs); everything smaller goes in one call per network after its backward pass, which sits on the critical path
    LARGE = int(os.environ.get("SG2_DP_LARGE", str(8 << 20)))

    def __init__(self, net, with_ema=False):
        self.params = [p for p in net.parameters()]
        dev = self.params[0].device
        sizes = [p.numel() for p in self.params]
        pad = lambda n: -(-n // 8) * 8           # keep every fp32 view 32-byte (bf16 mirror 16-byte, TMA) aligned
        # placement: the small parameters (BatchNorm, linear, biases, logit convs) first, as one contiguous head region,
        # then the conv weights — so that each conv weight AND the whole head are contiguous ranges (per-layer
        # all-reduce / Adam while backward is still running, one call for the rest).
        # Conv weights of at least LARGE elements come last: in a data-parallel run each of those is all-reduced on its
        # own as soon as its wgrad is done, everything before them (small params + small conv weights) in one call.
        offs, total = [None] * len(sizes), 0
        cls = lambda p, n: 0 if not _is_ohwi(p) else (1 if n < self.LARGE else 2)
        for want in (0, 1, 2):
            for i, (p, n) in enumerate(zip(self.params, sizes)):
                if cls(p, n) == want:
                    offs[i] = total
                    total += pad(n)
            if want == 0:
                self.head_n = total
            if want == 1:
                self.small_n = total
        self.n = total
        self.offs = offs
        self.range_of = {p: (o, pad(n)) for p, o, n in zip(self.params, offs, sizes)}
        self.flat = torch.zeros(total, device=dev, dtype=torch.float32)
        self.flat16 = torch.zeros(total, device=dev, dtype=torch.bfloat16)
        self.grad = torch.zeros_like(self.flat)
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.views = {}
        with torch.no_grad():
            for p, o, n in zip(self.params, offs, sizes):
                if _is_ohwi(p):
                    Co, Ci, kh, kw = p.shape
                    store = self.flat[o:o + n].view(Co, kh, kw, Ci)
                    store.copy_(p.detach().permute(0, 2, 3, 1))
                    p.data = store.permute(0, 3, 1, 2)
                    gstore = self.grad[o:o + n].view(Co, kh, kw, Ci)
                    self.views[p] = gstore.permute(0, 3, 1, 2)
                    p._sg2_ohwi = store.view(Co, kh * kw, Ci)
                    p._sg2_wpk = self.flat16[o:o + n].view(Co, kh * kw, Ci)
                    p._sg2_dw = gstore.view(Co, kh * kw, Ci)
                else:
                    self.flat[o:o + n].copy_(p.detach().reshape(-1))
                    p.data = self.flat[o:o + n].view(p.shape)
                    self.views[p] = self.grad[o:o + n].view(p.shape)
        ops.f32_to_bf16(self.flat, out=self.flat16)
        self.avg = self.flat.clone() if with_ema else None     # trainer.py:494 copy_G_params
        self.step = torch.zeros(1, device=dev, dtype=torch.int32)
        self.bc = torch.zeros(2, device=dev, dtype=torch.float32)

    def adam(self, lr, beta1=0.5, beta2=0.999, eps=1e-8, ema_decay=0.999):
        """One optimiser step over the whole bucket."""
        self.adam_tick(beta1, beta2)
        self.adam_range(0, self.n, lr, beta1, beta2, eps, ema_decay)
        self.dirty()

    def adam_tick(self, beta1=0.5, beta2=0.999):
        """Advance the device-side step counter / bias corrections: once per optimiser step, before any adam_range()."""
        ops._call("sg2_adam_tick", 1, _p(self.step), _p(self.bc), beta1, beta2, _st())

    def adam_range(self, o, n, lr, beta1=0.5, beta2=0.999, eps=1e-8, ema_decay=0.999):
        """Adam (+EMA, + bf16 mirror) on elements [o, o+n) of the bucket, on the current stream."""
        sl = slice(o, o + n)
        ops._call("sg2_adam_ema", 1, _p(self.flat[sl]), _p(self.grad[sl]), _p(self.m[sl]), _p(self.v[sl]),
                  _p(self.avg[sl]) if self.avg is not None else None, n, lr, beta1, beta2, eps, _p(self.bc), ema_decay,
                  _p(self.flat16[sl]), _st())

    def dirty(self):
        """The Adam kernel wrote the weights behind torch's back: invalidate the cached bf16 operand packs."""
        for p in self.params:
            p._sg2_version = getattr(p, "_sg2_version", 0) + 1

    def refresh(self):
        """Call after writing the parameters from outside the fused kernels (load_state_dict, `p.data.copy_`, an EMA
        swap through load_params, weights_init): re-derives the bf16 mirror from the fp32 masters and invalidates every
        cached operand pack."""
        ops.f32_to_bf16(self.flat, out=self.flat16)
        self.dirty()

    def swap_ema(self):
        """Exchange the live generator weights with the EMA shadow (what the reference does around its snapshot images
        with copy_G_params / load_params, trainer.py:592-601); call again to swap back."""
        if self.avg is None:
            raise RuntimeError("this bucket keeps no EMA shadow")
        tmp = self.flat.clone()
        self.flat.copy_(self.avg)
        self.avg.copy_(tmp)
        self.refresh()

    def ema_params(self):
        """EMA weights as a list shaped like net.parameters() (what trainer.py:256 load_params() copies in)."""
        out = []
        for p, o in zip(self.params, self.offs):
            n = p.numel()
            if _is_ohwi(p):
                Co, Ci, kh, kw = p.shape
                out.append(self.avg[o:o + n].view(Co, kh, kw, Ci).permute(0, 3, 1, 2))
            else:
                out.append(self.avg[o:o + n].view(p.shape))
        return out


class FusedTrainer:
    def __init__(self, netG, netsD, cfg, lr_g=None, lr_d=None, all_reduce=None, precision=None):
        """precision: None (config.PRECISION / what the networks were set to), 'bf16' or 'fp32' (fp32-accurate mode)."""
        self.netG, self.netsD = netG, list(netsD)
        if precision is not None:
            for net in [netG] + list(netsD):
                net.set_precision(precision)
        self.cfg = cfg
        c = cfg.TRAIN.COEFF
        self.uncond, self.cal, self.kl = float(c.UNCOND_LOSS), float(c.CAL_LOSS), float(c.KL)
        if self.uncond <= 0:
            raise NotImplementedError("UNCOND_LOSS == 0 is not used by any reference cfg")
        if float(getattr(c, "COLOR_LOSS", 0.0) or 0.0) > 0:
            # train_Gnet's colour-consistency terms (trainer.py:454-477); every reference cfg sets COLOR_LOSS: 0.0
            raise NotImplementedError("COLOR_LOSS > 0 (colour-consistency terms, trainer.py:454-477) is not implemented")
        self.lr_g = float(cfg.TRAIN.GENERATOR_LR if lr_g is None else lr_g)
        self.lr_d = float(cfg.TRAIN.DISCRIMINATOR_LR if lr_d is None else lr_d)
        self.G = netG.engine()
        self.Ds = [d.engine() for d in self.netsD]
        self.precise = self.G.precise
        if any(d.precise != self.precise for d in self.Ds):
            raise RuntimeError("sg2b200: G and D engines must run in the same precision")
        self.bG = FlatBucket(netG, with_ema=True)
        self.bD = [FlatBucket(d) for d in self.netsD]
        for eng in [self.G] + self.Ds:
            eng.set_auto_refresh(False)       # the buckets track every weight update themselves (dirty / refresh)
        self.all_reduce = all_reduce          # callable(flat_grad_tensor, chan) or None (single GPU)
        # Data parallel: (1) the persistent conv grids leave SG2_SM_RESERVE SMs (default 8) to NCCL's CTAs, so that the
        # per-layer all-reduces issued on the side streams advance while backward is still running instead of only in the
        # gaps between kernels; (2) SG2_GRAD_WIRE=bf16 halves the bytes on NVLink (468 -> 234 MB per step): the slice is
        # rounded to bf16, averaged, and widened back for Adam. Default fp32: the all-reduce is then exactly DDP's.
        self.wire_bf16 = all_reduce is not None and os.environ.get("SG2_GRAD_WIRE", "fp32") == "bf16"
        if all_reduce is not None:
            from . import _lib
            _lib.call("sg2_set_sm_reserve", int(os.environ.get("SG2_SM_RESERVE", "8")))
            if "SG2_PAIR" not in os.environ:
                # the CTA-pair kernels' cure (cluster barrier before the two-SM TMEM allocation) was stress-tested on one
                # GPU only; every 2 / 4 / 8-GPU line and the 2-GPU parity test of the round ran with them off
                _lib.call("sg2_set_pair_kernels", 0)
        self.concurrent = os.environ.get("SG2_CONCURRENT", "1") != "0"   # one stream per discriminator (see step())
        self.batched_d = os.environ.get("SG2_BATCHED_D", "1") != "0"     # real/wrong/fake D passes as one 3B pass
        # per-layer Adam (+ re-pack) on the wgrad side streams while backward is still running; data parallel: the large
        # layers (>= 32 MB of gradient) are all-reduced one by one as they complete, the rest in one call per network
        # (one small collective per layer measured slower: 11.7 vs 11.3 ms/step on 2 GPUs).
        self.layerwise = os.environ.get("SG2_LAYERWISE_OPT", "1") != "0"
        dev = self.bG.flat.device
        self.dev = dev
        # loss scalars: errD[i], errG_total, kl, cal
        self.losses = torch.zeros(len(self.Ds) + 3, device=dev, dtype=torch.float32)
        self._tables = {}

    # ------------------------------------------------------------------ state (checkpoint / resume, parity tests)
    def snapshot(self):
        """Everything a step reads and writes, cloned: flat parameters, Adam moments and step counters, the EMA shadow,
        BatchNorm running statistics (what the reference checkpoints with save_model plus the optimiser state)."""
        snap = {"buckets": [], "buffers": []}
        for b in [self.bG] + self.bD:
            snap["buckets"].append({k: getattr(b, k).clone() for k in ("flat", "m", "v", "step", "bc")}
                                   | ({"avg": b.avg.clone()} if b.avg is not None else {}))
        for net in [self.netG] + self.netsD:
            snap["buffers"].append([t.detach().clone() for t in net.buffers()])
        return snap

    def restore(self, snap):
        for b, sb in zip([self.bG] + self.bD, snap["buckets"]):
            for k, t in sb.items():
                getattr(b, k).copy_(t)
            b.refresh()
        for net, bufs in zip([self.netG] + self.netsD, snap["buffers"]):
            for t, src in zip(net.buffers(), bufs):
                t.copy_(src)
        # bring every cached operand pack up to date NOW (a captured graph re-packs a layer only after updating it)
        for eng in [self.G] + self.Ds:
            for op in eng.conv_ops():
                op.packs()

    # ------------------------------------------------------------------ helpers
    def _reduce(self, bucket, o, n, chan):
        """Average gradient elements [o, o+n) of the bucket over the ranks (in place)."""
        g = bucket.grad[o:o + n]
        if not self.wire_bf16:
            self.all_reduce(g, chan)
            return
        if getattr(bucket, "grad16", None) is None:
            bucket.grad16 = torch.empty(bucket.n, device=bucket.grad.device, dtype=torch.bfloat16)
        g16 = bucket.grad16[o:o + n]
        ops.f32_to_bf16(g, out=g16)
        self.all_reduce(g16, chan)
        ops._call("sg2_bf16_to_f32", 1, _p(g16), _p(g), n, _st())

    def _layerwise(self, bucket, lr, chan=0):
        """-> (on_ready, finish): all-reduce + Adam of each conv weight as soon as its wgrad is done (on the wgrad side
        stream, overlapping the rest of backward), then the small parameters and any leftover in finish()."""
        bucket.adam_tick()
        done = set()
        dp = self.all_reduce is not None

        def ready(w):
            o, n = bucket.range_of[w]
            if dp:
                if o < bucket.small_n:
                    return                       # small layer: reduced + updated with the rest in finish()
                self._reduce(bucket, o, n, chan)
            bucket.adam_range(o, n, lr)
            done.add(w)

        def repack(op):
            # the layer's master was just updated (ready) and its dgrad has been issued: refresh its bf16 operands now,
            # on the side stream, instead of lazily on the critical path of the next forward
            w = op.weight
            if w in done:
                w._sg2_version = getattr(w, "_sg2_version", 0) + 1
                op.packs()
                repacked.add(w)

        def finish():
            if dp:
                self._reduce(bucket, 0, bucket.small_n, chan)
                bucket.adam_range(0, bucket.small_n, lr)
            else:
                bucket.adam_range(0, bucket.head_n, lr)
            for w in bucket.params:
                o = bucket.range_of[w][0]
                if w not in done and o >= (bucket.small_n if dp else bucket.head_n):
                    ready(w)
            for w in bucket.params:
                if w not in repacked:
                    w._sg2_version = getattr(w, "_sg2_version", 0) + 1

        repacked = set()
        ready.repack = repack
        return ready, finish

    def _bce(self, probs, targets, weights, loss_slot):
        """probs (nvec, B) -> dprobs (nvec, B); adds sum_v w_v * BCE(probs[v], t_v) to loss_slot."""
        nvec, B = probs.shape
        dprobs = torch.empty_like(probs)
        key = (tuple(targets), tuple(weights))
        tw = self._tables.get(key)
        if tw is None:
            tw = (torch.tensor(targets, dtype=torch.float32, device=self.dev),
                  torch.tensor(weights, dtype=torch.float32, device=self.dev))
            self._tables[key] = tw
        ops._call("sg2_gan_bce", 1, _p(probs), _p(tw[0]), _p(tw[1]), nvec, B, _p(loss_slot), _p(dprobs), _st())
        return dprobs

    # ------------------------------------------------------------------ the step
    def _streams(self):
        if getattr(self, "_sD", None) is None:
            # the largest discriminator's update + G-step part is the longest branch of the step: its streams get the
            # higher priority so that its kernels are not queued behind the smaller discriminators' (SG2_PRIO=0: off)
            n = len(self.Ds)
            hi = -1 if os.environ.get("SG2_PRIO", "1") != "0" else 0
            prio = [hi if i == n - 1 and n > 1 else 0 for i in range(n)]
            self._sD = [torch.cuda.Stream(device=self.dev, priority=prio[i]) for i in range(n)]
            self._sW = [torch.cuda.Stream(device=self.dev, priority=(prio + [0])[i]) for i in range(n + 1)]  # wgrad side
            # per-layer optimiser work (unpack, all-reduce, Adam, re-pack) beside the wgrad stream (SG2_OPT_STREAM=0: off)
            two = os.environ.get("SG2_OPT_STREAM", "1") != "0"
            self._sO = [torch.cuda.Stream(device=self.dev, priority=(prio + [0])[i]) if two else None for i in range(n + 1)]
        return self._sD

    def step(self, z, emb, real, wrong, labels, eps=None, on_img=None):
        """z (B,Z) f32, emb (B,T) f32, real/wrong: lists of (B,3,S,S) f32 NCHW, labels (B,) int32 — all on the GPU.
        Returns the device tensor [errD_0.., errG_total, kl, cal] (no host sync). on_img(i, img): called on the current
        stream as soon as stage i's fake image has been issued (CapturedStep forks the Inception scoring there).

        Scheduling: the G forward runs on the current stream; the three discriminators are independent of one another
        (own weights, own optimiser, own image scale), so each D's update AND its part of the G step (forward on the
        live fake, backward to the image) run on their own stream; the current stream joins them before the G
        backward. Captured into a CUDA graph these become parallel branches."""
        nD = len(self.Ds)
        B = z.shape[0]
        main = torch.cuda.current_stream()
        streams = self._streams() if self.concurrent else [main] * nD
        ops.arena_reset(self.dev)
        self.losses.zero_()
        parts = torch.zeros(2 * nD, device=self.dev, dtype=torch.float32)    # per-D errG and cal (summed after the join)
        if eps is None:
            eps = torch.empty(B, self.G.E, device=self.dev, dtype=torch.float32).normal_()   # model.py:190-193
        # Work that does not depend on G runs on the D / side streams while the G forward occupies the main stream:
        # clearing the flat gradient buckets (conv weight gradients accumulate straight into them) and, for the batched
        # D update, the stem's im2col rows of real | wrong (one buffer per D; the fake third is filled after G).
        col3 = [None] * nD
        fork0 = torch.cuda.Event()
        fork0.record(main)
        for i in range(nD):
            st = streams[i]
            with torch.cuda.stream(st):
                if st is not main:
                    st.wait_event(fork0)
                if not ops.DETERMINISTIC:
                    self.bD[i].grad.zero_()       # red.global.add wgrads accumulate straight into the bucket
                if self.batched_d:
                    S = real[i].shape[2]
                    col3[i] = torch.empty((3, B * (S // 2) * (S // 2), 64), device=self.dev,
                                          dtype=torch.float32 if self.precise else torch.bfloat16)
                    ops.stem_im2col(real[i], out=col3[i][0])
                    ops.stem_im2col(wrong[i], out=col3[i][1])
        g_zeroed = None
        if self.concurrent and not ops.DETERMINISTIC:
            with torch.cuda.stream(self._sW[nD]):
                self._sW[nD].wait_event(fork0)
                self.bG.grad.zero_()
                g_zeroed = torch.cuda.Event()
                g_zeroed.record(self._sW[nD])
        # D_i's update needs mu and the stage-i image only: each discriminator's branch forks off the main stream as soon
        # as ITS image has been issued, so D64 / D128 run beside the later (bandwidth-bound, one-kernel-wide) generator
        # stages instead of beside D256 on the step's critical path (SG2_EARLY_FORK=1; off by default: measured 7.675 vs 7.62 ms/step — the small discriminators then compete with the generator chain)
        early = self.concurrent and os.environ.get("SG2_EARLY_FORK", "0") != "0"
        hook = {"mu3": None, "ev": [None] * nD}

        def on_mu(mu_):
            hook["mu3"] = mu_.repeat(3, 1) if self.batched_d else None

        def on_img_(i_, img_):
            if early and i_ < nD:
                hook["ev"][i_] = torch.cuda.Event()
                hook["ev"][i_].record(main)
            if on_img is not None:
                on_img(i_, img_)

        fake, mu, logvar, Tg = self.G.forward(z, emb, eps, True, on_mu=on_mu, on_img=on_img_)  # trainer.py:544
        mu3 = hook["mu3"]
        dmu = torch.empty_like(mu)
        dlogvar = torch.empty_like(logvar)
        kl = self.losses[nD + 1:nD + 2]
        ops._call("sg2_kl_loss", 1, _p(mu), _p(logvar), mu.numel(), self.kl, _p(kl), _p(dmu), _p(dlogvar), _st())
        fork = torch.cuda.Event()
        fork.record(main)
        dimgs, dcs, joins = [None] * nD, [None] * nD, []
        u = self.uncond
        for i, D in enumerate(self.Ds):
            st = streams[i]
            with torch.cuda.stream(st):
                if st is not main:
                    st.wait_event(hook["ev"][i] if hook["ev"][i] is not None else fork)
                    ops.arena_reset(self.dev)
                # ---------------- (2) update D_i, trainer.py:375-427
                bucket = self.bD[i]
                ready, fin = self._layerwise(bucket, self.lr_d, i) if (self.batched_d and self.layerwise) else (None, None)
                sink = GradSink(bucket.views, self._sW[i] if self.concurrent else None, prezeroed=True, on_ready=ready,
                                opt_stream=self._sO[i] if self.concurrent else None)
                sink.on_repack = ready.repack if ready is not None else None
                if self.batched_d:
                    # real | wrong | fake in ONE pass of 3B samples with per-sub-batch BatchNorm statistics: the same
                    # arithmetic as the reference's three passes (trainer.py:390-392), a third of the launches, and
                    # three times the GEMM rows for D's latency- and weight-bound layers.
                    ops.stem_im2col(fake[i], out=col3[i][2])
                    probs = torch.empty(2, 3 * B, device=self.dev, dtype=torch.float32)
                    _, _, _, T3 = D.forward((3 * B, fake[i].shape[2]), mu3, True, probs[0], probs[1], groups=3,
                                            stem_col=col3[i].view(1, 1, -1, 64), want_features=False)
                    # rows of probs.view(6, B): cond(real, wrong, fake), uncond(real, wrong, fake)
                    # targets: real -> 1,1 ; wrong -> cond 0, uncond 1 (trainer.py:400-401) ; fake -> 0,0
                    dprobs = self._bce(probs.view(6, B), (1, 0, 0, 1, 1, 0), (1, 1, 1, u, u, u), self.losses[i:i + 1])
                    dprobs = dprobs.view(2, 3 * B)
                    D.backward(T3, dprobs[0], dprobs[1], None, False, False, True, sink)
                    tapes = [T3]
                    # the fake third of the batched pass's im2col rows is exactly what the G step's D pass needs
                    fake_col = T3["stem"][0].view(3, -1, 64)[2].view(1, 1, -1, 64)
                else:
                    fake_col = None
                    tapes = []
                    probs = torch.empty(6, B, device=self.dev, dtype=torch.float32)
                    for k, img in enumerate((real[i], wrong[i], fake[i])):
                        _, _, _, T = D.forward(img, mu, True, probs[2 * k], probs[2 * k + 1], want_features=False)
                        tapes.append(T)
                    # targets: real -> 1,1 ; wrong -> cond 0, uncond 1 (trainer.py:400-401) ; fake -> 0,0
                    dprobs = self._bce(probs, (1, 1, 0, 1, 0, 0), (1, u, 1, u, 1, u), self.losses[i:i + 1])
                    for k, T in enumerate(tapes):
                        D.backward(T, dprobs[2 * k], dprobs[2 * k + 1], None, False, False, True, sink)
                sink.finish()
                del tapes
                if fin is not None:
                    fin()
                else:
                    if self.all_reduce is not None:
                        self._reduce(bucket, 0, bucket.n, i)
                    bucket.adam(self.lr_d)
                # ---------------- (3a) D_i's share of the G step, trainer.py:436-446 (updated D weights, live fake, mu)
                probs = torch.empty(2, B, device=self.dev, dtype=torch.float32)
                _, _, x_imm, T = D.forward(fake[i], mu, True, probs[0], probs[1], stem_col=fake_col,
                                           want_features=self.cal > 0)
                dprobs = self._bce(probs, (1, 1), (1, u), parts[i:i + 1])
                dx_imm = None
                if self.cal > 0:
                    ws = torch.empty(2 * B * B, device=self.dev, dtype=torch.float32)
                    dx_imm = torch.empty_like(x_imm)
                    ops._call("sg2_cal_loss", 3, _p(x_imm), _p(labels), B, x_imm.shape[1], _p(ws),
                              _p(parts[nD + i:nD + i + 1]), _p(dx_imm), _st())
                _, dimgs[i], dcs[i] = D.backward(T, dprobs[0], dprobs[1], dx_imm, True, True, False, None)
                if st is not main:
                    ev = torch.cuda.Event()
                    ev.record(st)
                    joins.append(ev)
        for ev in joins:
            main.wait_event(ev)
        # ---------------- (3b) G backward + update, trainer.py:480-488
        for dc in dcs:
            dmu.add_(dc)                         # mu is not detached in train_Gnet (trainer.py:438)
        if g_zeroed is not None:
            main.wait_event(g_zeroed)
        elif not ops.DETERMINISTIC:
            self.bG.grad.zero_()
        ready, fin = self._layerwise(self.bG, self.lr_g, nD) if self.layerwise else (None, None)
        sinkG = GradSink(self.bG.views, self._sW[nD] if self.concurrent else None, prezeroed=True, on_ready=ready,
                         opt_stream=self._sO[nD] if self.concurrent else None)
        sinkG.on_repack = ready.repack if ready is not None else None
        self.G.backward(Tg, dimgs, dmu, dlogvar, sinkG)
        sinkG.finish()
        if fin is not None:
            fin()                                # + EMA avg = 0.999 avg + 0.001 p (trainer.py:571-572)
        else:
            if self.all_reduce is not None:
                self._reduce(self.bG, 0, self.bG.n, nD)
            self.bG.adam(self.lr_g)
        # errG_total = sum_i errG_i + kl + sum_i cal_i (trainer.py:486)
        cal = self.losses[nD + 2:nD + 3]
        cal.add_(parts[nD:].sum())
        self.losses[nD:nD + 1].add_(parts[:nD].sum()).add_(kl).add_(cal)
        return self.losses


class CapturedStep:
    """The whole train step (noise draw, G forward, 3 D updates, G update, Adam, EMA — ~650 kernel launches) captured
    once into a CUDA graph and replayed per step: the launch-bound inner loop costs one cudaGraphLaunch instead of
    ~20 ms of Python/ctypes/driver work. Inputs live in static device buffers (`load()` copies a batch in)."""

    def __init__(self, trainer, batch_size, warmup=3, draw_noise=True, scorer=None, score_real=True):
        """draw_noise: the graph draws z ~ N(0,1) (trainer.py:542) and the reparameterisation eps (model.py:190-193) itself
        (Philox state advanced per replay); False: both come from the static buffers `noise` / `eps` filled by load()
        (parity tests replay the graph on given noise).
        scorer: an sg2b200.inception.INCEPTION_V3; the graph then also scores this step's last fake image and (score_real)
        the static real[-1] into `pred_fake` / `pool3_fake` / `pred_real` / `pool3_real`, what trainer.py:563-565
        computes. The scoring forks off the main stream once the last image is issued, runs on its own stream at normal
        priority (below the chain streams') and joins before the graph ends; it writes no training state."""
        self.tr = trainer
        cfg, dev = trainer.cfg, trainer.dev
        B = batch_size
        self.draw_noise = draw_noise
        self.scorer, self.score_real = scorer, score_real
        if scorer is not None:
            self._s_score = torch.cuda.Stream(device=dev, priority=0)
            self.pred_fake, self.pred_real = (torch.zeros(B, 1000, device=dev) for _ in range(2))
            self.pool3_fake, self.pool3_real = (torch.zeros(B, 2048, device=dev) for _ in range(2))
        self.noise = torch.zeros(B, cfg.GAN.Z_DIM, device=dev)
        self.eps = torch.zeros(B, cfg.GAN.EMBEDDING_DIM, device=dev)
        self.emb = torch.zeros(B, cfg.TEXT.DIMENSION, device=dev)
        sizes = [64 * 2 ** i for i in range(len(trainer.Ds))]
        self.real = [torch.zeros(B, 3, s, s, device=dev) for s in sizes]
        self.wrong = [torch.zeros(B, 3, s, s, device=dev) for s in sizes]
        self.labels = torch.zeros(B, device=dev, dtype=torch.int32)
        self.graph = None
        self.launches_per_step = 0
        self._warmup = warmup

    def load(self, emb, real, wrong, labels, non_blocking=True, z=None, eps=None):
        if z is not None:
            self.noise.copy_(z, non_blocking=non_blocking)
        if eps is not None:
            self.eps.copy_(eps, non_blocking=non_blocking)
        self.emb.copy_(emb, non_blocking=non_blocking)
        for d, s in zip(self.real, real):
            d.copy_(s, non_blocking=non_blocking)
        for d, s in zip(self.wrong, wrong):
            d.copy_(s, non_blocking=non_blocking)
        self.labels.copy_(labels, non_blocking=non_blocking)

    def _score(self, i, img):
        if i != len(self.tr.Ds) - 1:
            return
        fork = torch.cuda.Event()
        fork.record(torch.cuda.current_stream())
        s = self._s_score
        s.wait_event(fork)
        img.record_stream(s)
        with torch.cuda.stream(s):                                         # trainer.py:563-565
            self.scorer(img, out=(self.pred_fake, self.pool3_fake))
            if self.score_real:
                self.scorer(self.real[-1], out=(self.pred_real, self.pool3_real))
        self._scored = torch.cuda.Event()
        self._scored.record(s)

    def _body(self):
        hook = self._score if self.scorer is not None else None
        if self.draw_noise:
            self.noise.normal_(0, 1)                                       # trainer.py:542
            losses = self.tr.step(self.noise, self.emb, self.real, self.wrong, self.labels, on_img=hook)
        else:
            losses = self.tr.step(self.noise, self.emb, self.real, self.wrong, self.labels, eps=self.eps, on_img=hook)
        if hook is not None:
            torch.cuda.current_stream().wait_event(self._scored)
        return losses

    def capture(self):
        side = torch.cuda.Stream(device=self.tr.dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(self._warmup):                                  # eager steps: allocations, packs, caches
                self._body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        n0 = ops.launches()
        # the main branch (G forward, G backward) is on the step's critical path like the largest discriminator's
        hi = -1 if os.environ.get("SG2_PRIO_MAIN", "1") != "0" else 0
        with torch.cuda.graph(self.graph, stream=torch.cuda.Stream(device=self.tr.dev, priority=hi)):
            self.losses = self._body()
        self.launches_per_step = ops.launches() - n0
        return self

    def replay(self):
        self.graph.replay()
        return self.losses
