"""ORACLE — test infrastructure only (never imported by the product path).

A plain-PyTorch fp32 restatement of the reference's speech-conditioned StackGAN-v2 train step
(StackGAN_v2/model.py + trainer.py), written functionally over state dicts that use the
reference's own parameter names, so that reference checkpoints load unchanged.

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so this restatement is pinned
against the reference itself, imported from a checkout of it by oracle/make_golden.py; the outputs are
committed as tests/golden/*.npz and checked by tests/test_oracle.py (and, where a reference checkout is given
with SG2_REF, compared directly tensor-by-tensor).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this file.
"""
from dataclasses import dataclass, field

import torch
import torch.nn.functional as F


@dataclass
class Cfg:
    """The cfg keys the hot path reads (miscc/config.py:9-69; cfg/birds_3stages.yml)."""
    GF_DIM: int = 64
    DF_DIM: int = 64
    EMBEDDING_DIM: int = 128
    Z_DIM: int = 100
    R_NUM: int = 2
    TEXT_DIM: int = 1024
    BRANCH_NUM: int = 3
    UNCOND_LOSS: float = 1.0
    CAL_LOSS: float = 50.0
    KL: float = 2.0
    LR_G: float = 2e-4
    LR_D: float = 2e-4


BN_EPS, BN_MOM = 1e-5, 0.1

# bf16 emulation: when EMULATE_BF16 is set, every tensor the CUDA path stores in bf16 (conv operands, conv outputs,
# activation outputs) is rounded to bf16 here too, and so is the gradient that flows back through the same point (the
# CUDA backward stores dy / dx of every layer in bf16). The arithmetic in between stays fp32 (the tensor cores
# accumulate in fp32). Used by the GPU parity tests to separate "the kernels compute the same function" (tight
# tolerance vs the emulating oracle) from "bf16 storage vs the fp32 reference" (quantisation gap, reported).
# EMULATE_BF16 = "fwd": forward rounding only (straight-through gradients).
EMULATE_BF16 = False


class emulate_bf16:
    def __init__(self, on=True):
        self.on = on

    def __enter__(self):
        global EMULATE_BF16
        self.prev, EMULATE_BF16 = EMULATE_BF16, self.on

    def __exit__(self, *a):
        global EMULATE_BF16
        EMULATE_BF16 = self.prev


class _RoundBoth(torch.autograd.Function):
    """bf16 rounding of a stored tensor; the gradient stored at the same point is rounded too."""

    @staticmethod
    def forward(ctx, t):
        return t.bfloat16().float()

    @staticmethod
    def backward(ctx, g):
        return g.bfloat16().float()


def _q(t):
    if not EMULATE_BF16:
        return t
    if EMULATE_BF16 == "fwd" or not t.requires_grad:
        return t + (t.detach().bfloat16().float() - t.detach())
    return _RoundBoth.apply(t)


def _conv(x, w, **kw):
    return _q(F.conv2d(_q(x), _q(w), **kw))


# --------------------------------------------------------------------------------------------- building blocks
def glu(x):
    """model.py:112-122"""
    nc = x.size(1) // 2
    return _q(x[:, :nc] * torch.sigmoid(x[:, nc:]))


def _bn(x, sd, prefix, training):
    """nn.BatchNorm1d/2d (train: batch stats + running update, eval: running stats)."""
    if training:
        sd[prefix + ".num_batches_tracked"] += 1
    return F.batch_norm(x, sd[prefix + ".running_mean"], sd[prefix + ".running_var"], sd[prefix + ".weight"],
                        sd[prefix + ".bias"], training, BN_MOM, BN_EPS)


def _up_block(x, sd, prefix, training):
    """upBlock, model.py:133-140: nearest 2x, conv3x3, BN, GLU"""
    x = F.interpolate(x, scale_factor=2, mode="nearest")
    x = _conv(x, sd[prefix + ".1.weight"], padding=1)
    return glu(_bn(x, sd, prefix + ".2", training))


def _block3x3_glu(x, sd, prefix, training):
    """Block3x3_relu, model.py:144-150"""
    x = _conv(x, sd[prefix + ".0.weight"], padding=1)
    return glu(_bn(x, sd, prefix + ".1", training))


def _res_block(x, sd, prefix, training):
    """ResBlock, model.py:153-169"""
    h = _conv(x, sd[prefix + ".block.0.weight"], padding=1)
    h = glu(_bn(h, sd, prefix + ".block.1", training))
    h = _conv(h, sd[prefix + ".block.3.weight"], padding=1)
    h = _bn(h, sd, prefix + ".block.4", training)
    return _q(h + x)


def ca_net(sd, emb, eps, cfg):
    """CA_NET, model.py:172-200. eps is the N(0,1) draw the reference makes inside reparametrize."""
    x = glu(F.linear(emb, sd["ca_net.fc.weight"], sd["ca_net.fc.bias"]))
    mu, logvar = x[:, :cfg.EMBEDDING_DIM], x[:, cfg.EMBEDDING_DIM:]
    c = eps * torch.exp(0.5 * logvar) + mu
    return c, mu, logvar


def g_forward(sd, z, emb, eps, cfg, training=True):
    """G_NET.forward, model.py:327-354 -> ([img64, img128, img256][:BRANCH_NUM], mu, logvar)."""
    c, mu, logvar = ca_net(sd, emb, eps, cfg)
    ngf = cfg.GF_DIM * 16
    h = _q(F.linear(torch.cat((c, z), 1), sd["h_net1.fc.0.weight"]))      # model.py:227-233
    h = glu(_bn(h, sd, "h_net1.fc.1", training)).view(-1, ngf, 4, 4)
    for i in (1, 2, 3, 4):
        h = _up_block(h, sd, f"h_net1.upsample{i}", training)
    imgs = [torch.tanh(_conv(h, sd["img_net1.img.0.weight"], padding=1))]
    for stage in range(2, cfg.BRANCH_NUM + 1):
        p = f"h_net{stage}"
        s = h.size(2)
        cc = c.view(-1, cfg.EMBEDDING_DIM, 1, 1).repeat(1, 1, s, s)        # model.py:272-277
        if EMULATE_BF16:
            # the CUDA path folds the broadcast c_code channels into an fp32 per-sample bias (fp32 c, fp32 master
            # weights); only the h part goes through bf16 operands. Same function, different rounding points.
            w = sd[p + ".jointConv.0.weight"]
            e = cfg.EMBEDDING_DIM
            y = _q(F.conv2d(_q(h), _q(w[:, e:]), padding=1) + F.conv2d(cc, w[:, :e], padding=1))
            h = glu(_bn(y, sd, p + ".jointConv.1", training))
        else:
            h = _block3x3_glu(torch.cat((cc, h), 1), sd, p + ".jointConv", training)
        for r in range(cfg.R_NUM):
            h = _res_block(h, sd, f"{p}.residual.{r}", training)
        h = _up_block(h, sd, p + ".upsample", training)
        imgs.append(torch.tanh(_conv(h, sd[f"img_net{stage}.img.0.weight"], padding=1)))
    return imgs, mu, logvar


def _down(x, sd, conv, bn, training):
    x = _conv(x, sd[conv + ".weight"], stride=2, padding=1)
    if bn is not None:
        x = _bn(x, sd, bn, training)
    return _q(F.leaky_relu(x, 0.2))


def _block3x3_lrelu(x, sd, prefix, training):
    """Block3x3_leakRelu, model.py:358-365"""
    x = _conv(x, sd[prefix + ".0.weight"], padding=1)
    return _q(F.leaky_relu(_bn(x, sd, prefix + ".1", training), 0.2))


def d_forward(sd, img, c, which, cfg, training=True):
    """D_NET64/128/256.forward (which = 0/1/2), model.py:424-445, 473-496, 526-551
    -> ([cond (B,), uncond (B,)], x_immediate (B, 8*ndf*16))."""
    x = _down(img, sd, "img_code_s16.0", None, training)                   # model.py:380-398
    x = _down(x, sd, "img_code_s16.2", "img_code_s16.3", training)
    x = _down(x, sd, "img_code_s16.5", "img_code_s16.6", training)
    x = _down(x, sd, "img_code_s16.8", "img_code_s16.9", training)
    if which == 1:
        x = _down(x, sd, "img_code_s32.0", "img_code_s32.1", training)
        x = _block3x3_lrelu(x, sd, "img_code_s32_1", training)
    elif which == 2:
        x = _down(x, sd, "img_code_s32.0", "img_code_s32.1", training)
        x = _down(x, sd, "img_code_s64.0", "img_code_s64.1", training)
        x = _block3x3_lrelu(x, sd, "img_code_s64_1", training)
        x = _block3x3_lrelu(x, sd, "img_code_s64_2", training)
    x_immediate = x.reshape(x.shape[0], -1)
    cc = c.view(-1, cfg.EMBEDDING_DIM, 1, 1).repeat(1, 1, 4, 4)
    h = _block3x3_lrelu(torch.cat((_q(cc), x), 1), sd, "jointConv", training)
    cond = torch.sigmoid(F.conv2d(h, sd["logits.0.weight"], sd["logits.0.bias"], stride=4))
    uncond = torch.sigmoid(F.conv2d(x, sd["uncond_logits.0.weight"], sd["uncond_logits.0.bias"], stride=4))
    return [cond.view(-1), uncond.view(-1)], x_immediate


# --------------------------------------------------------------------------------------------- losses
def kl_loss(mu, logvar):
    """trainer.py:54-58"""
    return torch.mean(mu.pow(2).add(logvar.exp()).mul(-1).add(1).add(logvar)).mul(-0.5)


def bce(p, target):
    """nn.BCELoss (trainer.py:499): mean, log clamped at -100"""
    return F.binary_cross_entropy(p, target)


def class_aware_loss(x, labels):
    """trainer.py:298-311 (mask built on device instead of a Python double loop; same values)."""
    bsz, fdim = x.shape
    scores = x @ x.t()
    lab = torch.as_tensor(labels, device=x.device)
    pair = (lab[:, None] == lab[None, :]) & ~torch.eye(bsz, dtype=torch.bool, device=x.device)
    if int(pair.sum()) > 0:
        return torch.clamp(scores.mean() - scores[pair].mean(), min=0).div(fdim).reshape(1)
    return torch.zeros(1, device=x.device)


# --------------------------------------------------------------------------------------------- state dicts
def _orthogonal_(w):
    torch.nn.init.orthogonal_(w, 1.0)
    return w


def _bn_entries(sd, prefix, n):
    sd[prefix + ".weight"] = torch.empty(n).normal_(1.0, 0.02)
    sd[prefix + ".bias"] = torch.zeros(n)
    sd[prefix + ".running_mean"] = torch.zeros(n)
    sd[prefix + ".running_var"] = torch.ones(n)
    sd[prefix + ".num_batches_tracked"] = torch.zeros((), dtype=torch.long)


def init_g_state(cfg):
    """Parameter/buffer dict of G_NET with the reference's names, shapes, ORDER and weights_init
    (model.py:301-325; trainer.py:65-75)."""
    sd = {}
    e, ngf = cfg.EMBEDDING_DIM, cfg.GF_DIM * 16
    sd["ca_net.fc.weight"] = _orthogonal_(torch.empty(e * 4, cfg.TEXT_DIM))
    sd["ca_net.fc.bias"] = torch.zeros(e * 4)
    sd["h_net1.fc.0.weight"] = _orthogonal_(torch.empty(ngf * 4 * 4 * 2, cfg.Z_DIM + e))
    _bn_entries(sd, "h_net1.fc.1", ngf * 4 * 4 * 2)
    ch = ngf
    for i in (1, 2, 3, 4):
        sd[f"h_net1.upsample{i}.1.weight"] = _orthogonal_(torch.empty(ch, ch, 3, 3))
        _bn_entries(sd, f"h_net1.upsample{i}.2", ch)
        ch //= 2
    sd["img_net1.img.0.weight"] = _orthogonal_(torch.empty(3, ch, 3, 3))
    for stage in range(2, cfg.BRANCH_NUM + 1):
        p = f"h_net{stage}"
        sd[p + ".jointConv.0.weight"] = _orthogonal_(torch.empty(ch * 2, ch + e, 3, 3))
        _bn_entries(sd, p + ".jointConv.1", ch * 2)
        for r in range(cfg.R_NUM):
            sd[f"{p}.residual.{r}.block.0.weight"] = _orthogonal_(torch.empty(ch * 2, ch, 3, 3))
            _bn_entries(sd, f"{p}.residual.{r}.block.1", ch * 2)
            sd[f"{p}.residual.{r}.block.3.weight"] = _orthogonal_(torch.empty(ch, ch, 3, 3))
            _bn_entries(sd, f"{p}.residual.{r}.block.4", ch)
        sd[p + ".upsample.1.weight"] = _orthogonal_(torch.empty(ch, ch, 3, 3))
        _bn_entries(sd, p + ".upsample.2", ch)
        ch //= 2
        sd[f"img_net{stage}.img.0.weight"] = _orthogonal_(torch.empty(3, ch, 3, 3))
    return sd


def init_d_state(cfg, which):
    """Parameter/buffer dict of D_NET64/128/256 (which = 0/1/2), model.py:402-551."""
    sd = {}
    ndf, e = cfg.DF_DIM, cfg.EMBEDDING_DIM
    sd["img_code_s16.0.weight"] = _orthogonal_(torch.empty(ndf, 3, 4, 4))
    for idx, (ci, co) in zip((2, 5, 8), ((ndf, ndf * 2), (ndf * 2, ndf * 4), (ndf * 4, ndf * 8))):
        sd[f"img_code_s16.{idx}.weight"] = _orthogonal_(torch.empty(co, ci, 4, 4))
        _bn_entries(sd, f"img_code_s16.{idx + 1}", co)
    if which >= 1:
        sd["img_code_s32.0.weight"] = _orthogonal_(torch.empty(ndf * 16, ndf * 8, 4, 4))
        _bn_entries(sd, "img_code_s32.1", ndf * 16)
    if which == 1:
        sd["img_code_s32_1.0.weight"] = _orthogonal_(torch.empty(ndf * 8, ndf * 16, 3, 3))
        _bn_entries(sd, "img_code_s32_1.1", ndf * 8)
    if which == 2:
        sd["img_code_s64.0.weight"] = _orthogonal_(torch.empty(ndf * 32, ndf * 16, 4, 4))
        _bn_entries(sd, "img_code_s64.1", ndf * 32)
        sd["img_code_s64_1.0.weight"] = _orthogonal_(torch.empty(ndf * 16, ndf * 32, 3, 3))
        _bn_entries(sd, "img_code_s64_1.1", ndf * 16)
        sd["img_code_s64_2.0.weight"] = _orthogonal_(torch.empty(ndf * 8, ndf * 16, 3, 3))
        _bn_entries(sd, "img_code_s64_2.1", ndf * 8)
    sd["logits.0.weight"] = _orthogonal_(torch.empty(1, ndf * 8, 4, 4))
    sd["logits.0.bias"] = torch.empty(1).uniform_(-1, 1) * (1.0 / (ndf * 8 * 16)) ** 0.5   # Conv2d default bias init
    sd["jointConv.0.weight"] = _orthogonal_(torch.empty(ndf * 8, ndf * 8 + e, 3, 3))
    _bn_entries(sd, "jointConv.1", ndf * 8)
    sd["uncond_logits.0.weight"] = _orthogonal_(torch.empty(1, ndf * 8, 4, 4))
    sd["uncond_logits.0.bias"] = torch.empty(1).uniform_(-1, 1) * (1.0 / (ndf * 8 * 16)) ** 0.5
    return sd


def is_param(key):
    return not (key.endswith("running_mean") or key.endswith("running_var") or key.endswith("num_batches_tracked"))


def param_keys(sd):
    return [k for k in sd if is_param(k)]


# --------------------------------------------------------------------------------------------- train step
def synthetic_batch(cfg, batch, seed=1234, device="cpu", n_classes=4):
    """Synthetic inputs of SURVEY.md section 8(d): z, speech embedding, real/wrong image pyramids, labels."""
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(batch, cfg.Z_DIM, generator=g)
    emb = torch.randn(batch, cfg.TEXT_DIM, generator=g)
    eps = torch.randn(batch, cfg.EMBEDDING_DIM, generator=g)
    real, wrong = [], []
    for i in range(cfg.BRANCH_NUM):
        s = 64 * 2 ** i
        real.append(torch.rand(batch, 3, s, s, generator=g) * 2 - 1)
        wrong.append(torch.rand(batch, 3, s, s, generator=g) * 2 - 1)
    labels = torch.randint(0, n_classes, (batch,), generator=g)
    mv = lambda t: t.to(device)
    return dict(z=mv(z), emb=mv(emb), eps=mv(eps), real=[mv(t) for t in real], wrong=[mv(t) for t in wrong],
                labels=labels.tolist())


class OracleTrainer:
    """condGANTrainer.train's inner loop (trainer.py:529-572 minus Inception), fp32, any device.

    step(batch) = G forward -> train_Dnet x BRANCH_NUM -> train_Gnet -> EMA, with torch.optim.Adam.
    Returns every loss and (optionally) every gradient so parity tests can compare them."""

    def __init__(self, cfg, g_state=None, d_states=None, device="cpu"):
        self.cfg = cfg
        self.device = torch.device(device)
        mv = lambda sd: {k: v.clone().to(self.device) for k, v in sd.items()}
        self.g = mv(g_state if g_state is not None else init_g_state(cfg))
        self.ds = [mv(d_states[i] if d_states is not None else init_d_state(cfg, i)) for i in range(cfg.BRANCH_NUM)]
        for sd in [self.g] + self.ds:
            for k in param_keys(sd):
                sd[k].requires_grad_(True)
        self.opt_g = torch.optim.Adam([self.g[k] for k in param_keys(self.g)], lr=cfg.LR_G, betas=(0.5, 0.999))
        self.opt_d = [torch.optim.Adam([sd[k] for k in param_keys(sd)], lr=cfg.LR_D, betas=(0.5, 0.999))
                      for sd in self.ds]
        self.avg_g = [self.g[k].detach().clone() for k in param_keys(self.g)]   # trainer.py:494

    def step(self, batch, keep_grads=False, update=True):
        cfg = self.cfg
        out = {}
        bsz = batch["z"].shape[0]
        ones = torch.ones(bsz, device=self.device, dtype=batch["z"].dtype)     # float64 runs: targets in float64 too
        zeros = torch.zeros(bsz, device=self.device, dtype=batch["z"].dtype)
        fake, mu, logvar = g_forward(self.g, batch["z"], batch["emb"], batch["eps"], cfg, True)   # trainer.py:544
        out["fake"], out["mu"], out["logvar"] = [f.detach() for f in fake], mu.detach(), logvar.detach()
        # ---- train_Dnet (trainer.py:375-427)
        out["errD"], out["d_logits"] = [], []
        grads_d = []
        for i, sd in enumerate(self.ds):
            for k in param_keys(sd):
                sd[k].grad = None
            rl, _ = d_forward(sd, batch["real"][i], mu.detach(), i, cfg)
            wl, _ = d_forward(sd, batch["wrong"][i], mu.detach(), i, cfg)
            fl, _ = d_forward(sd, fake[i].detach(), mu.detach(), i, cfg)
            err_real = bce(rl[0], ones) + cfg.UNCOND_LOSS * bce(rl[1], ones)
            err_wrong = bce(wl[0], zeros) + cfg.UNCOND_LOSS * bce(wl[1], ones)      # trainer.py:400-401
            err_fake = bce(fl[0], zeros) + cfg.UNCOND_LOSS * bce(fl[1], zeros)
            err = err_real + err_wrong + err_fake
            err.backward()
            out["errD"].append(err.detach())
            out["d_logits"].append([t.detach() for t in (rl + wl + fl)])
            if keep_grads:
                grads_d.append({k: sd[k].grad.detach().clone() for k in param_keys(sd)})
            if update:
                self.opt_d[i].step()
        # ---- train_Gnet (trainer.py:429-489)
        for k in param_keys(self.g):
            self.g[k].grad = None
        err_total = 0
        cal_total = 0
        out["g_logits"], out["x_active"] = [], []
        for i, sd in enumerate(self.ds):
            outputs, x_active = d_forward(sd, fake[i], mu, i, cfg)
            err_total = err_total + bce(outputs[0], ones) + cfg.UNCOND_LOSS * bce(outputs[1], ones)
            if cfg.CAL_LOSS > 0:
                cal_total = cal_total + class_aware_loss(x_active, batch["labels"])
            out["g_logits"].append([t.detach() for t in outputs])
            out["x_active"].append(x_active.detach())
        kl = kl_loss(mu, logvar) * cfg.KL
        err_total = err_total + kl + cal_total
        err_total.backward()
        out["kl"], out["errG_total"] = kl.detach(), err_total.detach().reshape(())
        out["cal"] = cal_total.detach() if torch.is_tensor(cal_total) else torch.zeros(1)
        if keep_grads:
            out["grads_g"] = {k: self.g[k].grad.detach().clone() for k in param_keys(self.g)}
            out["grads_d"] = grads_d
        if update:
            self.opt_g.step()
            for p, avg in zip((self.g[k] for k in param_keys(self.g)), self.avg_g):     # trainer.py:571-572
                avg.mul_(0.999).add_(p.detach(), alpha=0.001)
        return out
