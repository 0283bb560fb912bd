"""Inception-v3 scorer on the sg2b200 kernels: drop-in for the reference's INCEPTION_V3 (model.py:17-109), which the
reference trainer runs on fake_imgs[-1] and real_imgs[-1] every step (trainer.py:563-565) for the Inception Score, FID
and NLPP (trainer.py:88-159).

The module holds torchvision `Inception3` parameters under the reference's wrapper attribute `model` (same names,
shapes and order, AuxLogits included so the pretrained file loads strictly; AuxLogits never runs). It is forward-only
and always in eval mode: every BasicConv2d (conv, BatchNorm2d(eps=0.001) on running statistics, ReLU) is folded in
float64 on the host into one bf16 convolution with an fp32 bias and ReLU in the epilogue (sg2_conv2d_fprop). The fold
is redone whenever a parameter or buffer is written (load_state_dict, in-place updates). The branches of an Inception
block write into their channel slice of the block output, so there is no concatenation.

forward(img): img (B,3,S,S) fp32 CUDA in [-1, 1] -> (pred (B,1000) softmax, pool3 (B,2048)), fp32, no autograd graph.
Preprocessing as the reference: x*0.5+0.5, ImageNet mean / std, bilinear resize to 299x299 (align_corners=False), all
fused into the im2col stem of Conv2d_1a_3x3. Arithmetic: bf16 operands, fp32 accumulation, bf16 activations.

torchvision is not imported: the holders below reproduce its module tree.
"""
import os

import torch
from torch import nn

from . import ops

WEIGHTS_FILE = "inception_v3_google-1a9a5a14.pth"
BN_EPS = 0.001


class BasicConv2d(nn.Module):
    """Parameter holder of torchvision's BasicConv2d; (kh, kw, stride, ph, pw) is the geometry the kernels run."""

    def __init__(self, cin, cout, k, stride=1, pad=0):
        super().__init__()
        kh, kw = (k, k) if isinstance(k, int) else k
        ph, pw = (pad, pad) if isinstance(pad, int) else pad
        self.conv = nn.Conv2d(cin, cout, (kh, kw), stride=stride, padding=(ph, pw), bias=False)
        self.bn = nn.BatchNorm2d(cout, eps=BN_EPS)
        self.geo = (cin, cout, kh, kw, stride, ph, pw)


class InceptionA(nn.Module):
    def __init__(self, cin, pool_features):
        super().__init__()
        self.branch1x1 = BasicConv2d(cin, 64, 1)
        self.branch5x5_1 = BasicConv2d(cin, 48, 1)
        self.branch5x5_2 = BasicConv2d(48, 64, 5, pad=2)
        self.branch3x3dbl_1 = BasicConv2d(cin, 64, 1)
        self.branch3x3dbl_2 = BasicConv2d(64, 96, 3, pad=1)
        self.branch3x3dbl_3 = BasicConv2d(96, 96, 3, pad=1)
        self.branch_pool = BasicConv2d(cin, pool_features, 1)
        self.cout = 224 + pool_features

    def plan(self):
        # per branch, in order: (input, conv, output channel offset). input None: the block input, "t": the branch's
        # previous intermediate, "avg": the block input after avg-pool 3x3 s1 p1, "max": max-pool 3x3 s2 of the block
        # input (no conv); offset None: an intermediate, else the conv writes that channel slice of the block output
        return [[(None, "branch1x1", 0)],
                [(None, "branch5x5_1", None), ("t", "branch5x5_2", 64)],
                [(None, "branch3x3dbl_1", None), ("t", "branch3x3dbl_2", None), ("t", "branch3x3dbl_3", 128)],
                [("avg", "branch_pool", 224)]]


class InceptionB(nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.branch3x3 = BasicConv2d(cin, 384, 3, stride=2)
        self.branch3x3dbl_1 = BasicConv2d(cin, 64, 1)
        self.branch3x3dbl_2 = BasicConv2d(64, 96, 3, pad=1)
        self.branch3x3dbl_3 = BasicConv2d(96, 96, 3, stride=2)
        self.cout = 480 + cin

    def plan(self):
        return [[(None, "branch3x3", 0)],
                [(None, "branch3x3dbl_1", None), ("t", "branch3x3dbl_2", None), ("t", "branch3x3dbl_3", 384)],
                [("max", None, 480)]]


class InceptionC(nn.Module):
    def __init__(self, cin, c7):
        super().__init__()
        self.branch1x1 = BasicConv2d(cin, 192, 1)
        self.branch7x7_1 = BasicConv2d(cin, c7, 1)
        self.branch7x7_2 = BasicConv2d(c7, c7, (1, 7), pad=(0, 3))
        self.branch7x7_3 = BasicConv2d(c7, 192, (7, 1), pad=(3, 0))
        self.branch7x7dbl_1 = BasicConv2d(cin, c7, 1)
        self.branch7x7dbl_2 = BasicConv2d(c7, c7, (7, 1), pad=(3, 0))
        self.branch7x7dbl_3 = BasicConv2d(c7, c7, (1, 7), pad=(0, 3))
        self.branch7x7dbl_4 = BasicConv2d(c7, c7, (7, 1), pad=(3, 0))
        self.branch7x7dbl_5 = BasicConv2d(c7, 192, (1, 7), pad=(0, 3))
        self.branch_pool = BasicConv2d(cin, 192, 1)
        self.cout = 768

    def plan(self):
        return [[(None, "branch1x1", 0)],
                [(None, "branch7x7_1", None), ("t", "branch7x7_2", None), ("t", "branch7x7_3", 192)],
                [(None, "branch7x7dbl_1", None), ("t", "branch7x7dbl_2", None), ("t", "branch7x7dbl_3", None),
                 ("t", "branch7x7dbl_4", None), ("t", "branch7x7dbl_5", 384)],
                [("avg", "branch_pool", 576)]]


class InceptionD(nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.branch3x3_1 = BasicConv2d(cin, 192, 1)
        self.branch3x3_2 = BasicConv2d(192, 320, 3, stride=2)
        self.branch7x7x3_1 = BasicConv2d(cin, 192, 1)
        self.branch7x7x3_2 = BasicConv2d(192, 192, (1, 7), pad=(0, 3))
        self.branch7x7x3_3 = BasicConv2d(192, 192, (7, 1), pad=(3, 0))
        self.branch7x7x3_4 = BasicConv2d(192, 192, 3, stride=2)
        self.cout = 512 + cin

    def plan(self):
        return [[(None, "branch3x3_1", None), ("t", "branch3x3_2", 0)],
                [(None, "branch7x7x3_1", None), ("t", "branch7x7x3_2", None), ("t", "branch7x7x3_3", None),
                 ("t", "branch7x7x3_4", 320)],
                [("max", None, 512)]]


class InceptionE(nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.branch1x1 = BasicConv2d(cin, 320, 1)
        self.branch3x3_1 = BasicConv2d(cin, 384, 1)
        self.branch3x3_2a = BasicConv2d(384, 384, (1, 3), pad=(0, 1))
        self.branch3x3_2b = BasicConv2d(384, 384, (3, 1), pad=(1, 0))
        self.branch3x3dbl_1 = BasicConv2d(cin, 448, 1)
        self.branch3x3dbl_2 = BasicConv2d(448, 384, 3, pad=1)
        self.branch3x3dbl_3a = BasicConv2d(384, 384, (1, 3), pad=(0, 1))
        self.branch3x3dbl_3b = BasicConv2d(384, 384, (3, 1), pad=(1, 0))
        self.branch_pool = BasicConv2d(cin, 192, 1)
        self.cout = 2048

    def plan(self):   # the 1x3 and 3x1 convs both read the branch's previous output (torchvision's torch.cat of the two)
        return [[(None, "branch1x1", 0)],
                [(None, "branch3x3_1", None), ("t", "branch3x3_2a", 320), ("t", "branch3x3_2b", 704)],
                [(None, "branch3x3dbl_1", None), ("t", "branch3x3dbl_2", None), ("t", "branch3x3dbl_3a", 1088),
                 ("t", "branch3x3dbl_3b", 1472)],
                [("avg", "branch_pool", 1856)]]


class InceptionAux(nn.Module):
    """Holder only: the pretrained file has it, the scorer never runs it."""

    def __init__(self, cin, num_classes):
        super().__init__()
        self.conv0 = BasicConv2d(cin, 128, 1)
        self.conv1 = BasicConv2d(128, 768, 5)
        self.fc = nn.Linear(768, num_classes)


class Inception3(nn.Module):
    """torchvision.models.Inception3(aux_logits=True, transform_input=False)'s parameter tree."""

    STEM = ("Conv2d_1a_3x3", "Conv2d_2a_3x3", "Conv2d_2b_3x3", "maxpool", "Conv2d_3b_1x1", "Conv2d_4a_3x3", "maxpool")
    BLOCKS = ("Mixed_5b", "Mixed_5c", "Mixed_5d", "Mixed_6a", "Mixed_6b", "Mixed_6c", "Mixed_6d", "Mixed_6e",
              "Mixed_7a", "Mixed_7b", "Mixed_7c")

    def __init__(self, num_classes=1000):
        super().__init__()
        self.Conv2d_1a_3x3 = BasicConv2d(3, 32, 3, stride=2)
        self.Conv2d_2a_3x3 = BasicConv2d(32, 32, 3)
        self.Conv2d_2b_3x3 = BasicConv2d(32, 64, 3, pad=1)
        self.Conv2d_3b_1x1 = BasicConv2d(64, 80, 1)
        self.Conv2d_4a_3x3 = BasicConv2d(80, 192, 3)
        self.Mixed_5b = InceptionA(192, 32)
        self.Mixed_5c = InceptionA(256, 64)
        self.Mixed_5d = InceptionA(288, 64)
        self.Mixed_6a = InceptionB(288)
        self.Mixed_6b = InceptionC(768, 128)
        self.Mixed_6c = InceptionC(768, 160)
        self.Mixed_6d = InceptionC(768, 160)
        self.Mixed_6e = InceptionC(768, 192)
        self.AuxLogits = InceptionAux(768, num_classes)
        self.Mixed_7a = InceptionD(768)
        self.Mixed_7b = InceptionE(1280)
        self.Mixed_7c = InceptionE(2048)
        self.fc = nn.Linear(2048, num_classes)


def default_weight_paths():
    """Where the weights are looked for when no path is given: $SG2_INCEPTION_WEIGHTS, then the file the reference's
    model_zoo.load_url leaves in the torch hub cache."""
    paths = []
    if os.environ.get("SG2_INCEPTION_WEIGHTS"):
        paths.append(os.environ["SG2_INCEPTION_WEIGHTS"])
    paths.append(os.path.join(torch.hub.get_dir(), "checkpoints", WEIGHTS_FILE))
    return paths


def fold_bn(w, gamma, beta, mean, var, eps=BN_EPS):
    """conv(w) -> BN(eval) as one conv with a bias, in float64: (w * s, beta - mean * s), s = gamma / sqrt(var + eps)."""
    s = gamma.double() / torch.sqrt(var.double() + eps)
    return w.double() * s.view(-1, 1, 1, 1), beta.double() - mean.double() * s


def layer_plan(S=299):
    """Every convolution the scorer runs at an S x S input (S = 299 after the resize): list of dicts with the layer name,
    geometry, input size and MACs per image. Conv2d_1a_3x3 runs as a K = 32 GEMM over the stem's im2col rows."""
    net = Inception3()
    out = []
    H = S

    def add(name, m, H, W):
        cin, cout, kh, kw, st, ph, pw = m.geo
        Ho, Wo = ops.conv2d_out_hw(H, W, kh, kw, st, ph, pw)
        out.append(dict(name=name, cin=cin, cout=cout, kh=kh, kw=kw, stride=st, ph=ph, pw=pw, H=H, W=W, Ho=Ho, Wo=Wo,
                        macs=Ho * Wo * cout * cin * kh * kw))
        return Ho

    for name in Inception3.STEM:
        H = (H - 3) // 2 + 1 if name == "maxpool" else add(name, getattr(net, name), H, H)
    for bname in Inception3.BLOCKS:
        blk = getattr(net, bname)
        Hn = H
        for branch in blk.plan():
            h = H
            for src, conv, c0 in branch:
                if conv is None:
                    Hn = (H - 3) // 2 + 1
                    continue
                h2 = add(f"{bname}.{conv}", getattr(blk, conv), h if src == "t" else H, h if src == "t" else H)
                if c0 is None:
                    h = h2
                Hn = h2
        H = Hn
    return out


def utilisation_report(B, S=299):
    """Issued versus useful MMA rows (and columns) of every convolution at batch B, from sg2_conv2d_plan."""
    rows = []
    for L in layer_plan(S):
        if L["name"] == "Conv2d_1a_3x3":   # the stem GEMM: 1x1 over (B, 149, 149) pixels of K = 32
            p = ops.conv2d_plan(B, L["Ho"], L["Wo"], 32, L["cout"], 1, 1)
        else:
            p = ops.conv2d_plan(B, L["H"], L["W"], L["cin"], L["cout"], L["kh"], L["kw"], L["stride"], L["ph"], L["pw"])
        rows.append(dict(L, **p, row_use=p["useful_rows"] / p["issued_rows"], col_use=L["cout"] / p["issued_cols"]))
    return rows


class INCEPTION_V3(nn.Module):
    """Drop-in for the reference's INCEPTION_V3 (model.py:17-109) on the sg2b200 kernels.

    weights: path of a torchvision Inception-v3 state dict (inception_v3_google-1a9a5a14.pth); None: the first of
    default_weight_paths() that exists. Nothing is ever downloaded: FileNotFoundError names the paths tried.
    random_init=True: keep the random initialisation (tests), no file is read."""

    def __init__(self, weights=None, random_init=False):
        super().__init__()
        self.model = Inception3()
        if not random_init:
            paths = [weights] if weights is not None else default_weight_paths()
            path = next((p for p in paths if os.path.isfile(p)), None)
            if path is None:
                raise FileNotFoundError("Inception-v3 weights not found (nothing is downloaded); tried: " +
                                        ", ".join(paths) + ". Pass INCEPTION_V3(weights=path) or set "
                                        "SG2_INCEPTION_WEIGHTS.")
            sd = torch.load(path, map_location="cpu", weights_only=True)
            self.model.load_state_dict(sd)
        for p in self.parameters():
            p.requires_grad_(False)
        self.eval()
        self._fold_key = None
        self._packs = None

    # ---- folding
    def _key(self, dev):
        return (dev,) + tuple((t.data_ptr(), t._version) for t in self.model.state_dict(keep_vars=True).values())

    def _fold(self, dev):
        key = self._key(dev)
        if key == self._fold_key:
            return self._packs
        packs = {}
        for name, m in self.model.named_modules():
            if not isinstance(m, BasicConv2d) or name.startswith("AuxLogits"):
                continue
            w, b = fold_bn(m.conv.weight.detach().cpu(), m.bn.weight.detach().cpu(), m.bn.bias.detach().cpu(),
                           m.bn.running_mean.detach().cpu(), m.bn.running_var.detach().cpu(), m.bn.eps)
            w = w.permute(0, 2, 3, 1).reshape(w.shape[0], -1)           # [Cout][kh][kw][Cin]
            if name == "Conv2d_1a_3x3":                                  # K = 27 (ky, kx, c) -> 32: the stem's rows
                w = torch.cat([w, w.new_zeros(w.shape[0], 32 - w.shape[1])], 1)
            packs[name] = (w.to(torch.bfloat16).contiguous().to(dev), b.float().contiguous().to(dev))
        fc = self.model.fc
        packs["fc"] = (fc.weight.detach().float().contiguous().to(dev), fc.bias.detach().float().contiguous().to(dev))
        self._packs, self._fold_key = packs, key
        return packs

    # ---- forward
    def _conv(self, packs, name, m, x, out=None, out_c0=0):
        cin, cout, kh, kw, st, ph, pw = m.geo
        B, H, W, _ = x.shape
        if out is None:
            Ho, Wo = ops.conv2d_out_hw(H, W, kh, kw, st, ph, pw)
            out = torch.empty((B, Ho, Wo, cout), device=x.device, dtype=torch.bfloat16)
        w, b = packs[name]
        return ops.conv2d_fprop(x, cin, w, b, out, cout, kh, kw, st, ph, pw, True, 0, out_c0)

    def _block(self, packs, bname, blk, x):
        B, H, W, _ = x.shape
        out = None
        for branch in blk.plan():
            t = x
            for src, conv, c0 in branch:
                if src == "max":
                    if out is None:
                        out = torch.empty((B, (H - 3) // 2 + 1, (W - 3) // 2 + 1, blk.cout), device=x.device,
                                          dtype=torch.bfloat16)
                    ops.maxpool3s2(x, out, c0)
                    continue
                m = getattr(blk, conv)
                inp = t if src == "t" else (ops.avgpool3s1(x) if src == "avg" else x)
                if c0 is None:
                    t = self._conv(packs, f"{bname}.{conv}", m, inp)
                else:
                    if out is None:
                        _, _, kh, kw, st, ph, pw = m.geo
                        Ho, Wo = ops.conv2d_out_hw(inp.shape[1], inp.shape[2], kh, kw, st, ph, pw)
                        out = torch.empty((B, Ho, Wo, blk.cout), device=x.device, dtype=torch.bfloat16)
                    self._conv(packs, f"{bname}.{conv}", m, inp, out, c0)
        return out

    def forward(self, img, out=None):
        """out: optional (pred, pool3) fp32 buffers to write (the captured train step's static outputs)."""
        if self.training:
            raise RuntimeError("sg2b200 INCEPTION_V3 is an eval-mode scorer (the reference scores in eval mode): "
                               "call .eval()")
        if not img.is_cuda:
            raise RuntimeError("sg2b200 kernels need CUDA tensors (there is no CPU fallback)")
        if img.dim() != 4 or img.shape[1] != 3 or img.shape[2] != img.shape[3]:
            raise RuntimeError(f"INCEPTION_V3: expected (B, 3, S, S) images, got {tuple(img.shape)}")
        with torch.no_grad():
            packs = self._fold(img.device)
            net = self.model
            x = ops.inception_stem(img.float().contiguous())
            w1, b1 = packs["Conv2d_1a_3x3"]            # K = 32 GEMM over the stem's im2col rows
            x = ops.conv2d_fprop(x, 32, w1, b1, torch.empty_like(x), 32, 1, 1)
            for name in Inception3.STEM[1:]:
                x = ops.maxpool3s2(x) if name == "maxpool" else self._conv(packs, name, getattr(net, name), x)
            for bname in Inception3.BLOCKS:
                x = self._block(packs, bname, getattr(net, bname), x)
            pred, pool3 = out if out is not None else (None, None)
            if out is not None and (pred.shape != (img.shape[0], 1000) or pool3.shape != (img.shape[0], 2048) or
                                    pred.dtype != torch.float32 or pool3.dtype != torch.float32):
                raise RuntimeError("INCEPTION_V3: out must be fp32 (B, 1000) and (B, 2048) buffers")
            pool3 = ops.global_avg(x, pool3)
            logits = ops.linear_fwd(pool3, None, packs["fc"][0], packs["fc"][1], out_bf16=False)
            return ops.softmax_rows(logits, pred), pool3
