"""ORACLE support — import the UNMODIFIED reference (StackGAN_v2/model.py, trainer.py) from a checkout of it.

Test infrastructure only. The reference needs `easydict` and `tensorboardX` (absent here): two in-memory shims
are installed before import (SURVEY.md section 8c). cfg is set by assignment (config.py:109 `yaml.load(f)`
raises under PyYAML 6). Nothing is copied from the reference; it is executed where it lies.

The repository does not ship the reference: callers must check `reference_available()`.
"""
import os
import sys
import types

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# $SG2_REF, or a checkout placed under baseline/_ref (git-ignored; never created by this repo: the reference is a
# Python source tree that must not be copied)
REF_CANDIDATES = [os.environ.get("SG2_REF", ""), os.path.join(_ROOT, "baseline", "_ref", "StackGAN_v2")]


def reference_dir():
    for d in REF_CANDIDATES:
        if d and os.path.isfile(os.path.join(d, "model.py")):
            return d
    return None


def reference_available():
    return reference_dir() is not None


class _EasyDict(dict):
    """Stand-in for easydict.EasyDict: attribute + item access, recursive dict conversion."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            setattr(self, k, v)

    def __setattr__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, _EasyDict):
            v = _EasyDict(v)
        super().__setitem__(k, v)

    __setitem__ = __setattr__

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


class _SummaryWriter:
    def __init__(self, *a, **k):
        pass

    def add_scalar(self, *a, **k):
        pass

    add_scalars = add_image = add_scalar

    def close(self):
        pass


def load_reference(cfg):
    """Import reference `model` and `trainer` with the global cfg set from an oracle Cfg. Returns (model, trainer, refcfg)."""
    d = reference_dir()
    if d is None:
        raise RuntimeError("reference not available")
    if "easydict" not in sys.modules:
        m = types.ModuleType("easydict")
        m.EasyDict = _EasyDict
        sys.modules["easydict"] = m
    if "tensorboardX" not in sys.modules:
        m = types.ModuleType("tensorboardX")
        m.SummaryWriter = _SummaryWriter
        sys.modules["tensorboardX"] = m
    if d not in sys.path:
        sys.path.insert(0, d)
    from miscc.config import cfg as rcfg
    rcfg.CUDA = False
    rcfg.TREE.BRANCH_NUM = cfg.BRANCH_NUM
    rcfg.GAN.GF_DIM = cfg.GF_DIM
    rcfg.GAN.DF_DIM = cfg.DF_DIM
    rcfg.GAN.EMBEDDING_DIM = cfg.EMBEDDING_DIM
    rcfg.GAN.Z_DIM = cfg.Z_DIM
    rcfg.GAN.R_NUM = cfg.R_NUM
    rcfg.GAN.B_CONDITION = True
    rcfg.TEXT.DIMENSION = cfg.TEXT_DIM
    rcfg.TRAIN.COEFF.UNCOND_LOSS = cfg.UNCOND_LOSS
    rcfg.TRAIN.COEFF.CAL_LOSS = cfg.CAL_LOSS
    rcfg.TRAIN.COEFF.KL = cfg.KL
    rcfg.TRAIN.COEFF.COLOR_LOSS = 0.0
    rcfg.TRAIN.GENERATOR_LR = cfg.LR_G
    rcfg.TRAIN.DISCRIMINATOR_LR = cfg.LR_D
    rcfg.TRAIN.LOG_INTERVAL = 10 ** 9
    import model as ref_model
    import trainer as ref_trainer
    return ref_model, ref_trainer, rcfg


def build_reference_trainer(cfg, batch_size):
    """A condGANTrainer wired the way trainer.train() does (trainer.py:491-520) without load_network()
    (which would download Inception weights, model.py:84-88)."""
    import torch
    import torch.nn as nn
    ref_model, ref_trainer, rcfg = load_reference(cfg)
    rcfg.TRAIN.BATCH_SIZE = batch_size
    t = ref_trainer.condGANTrainer.__new__(ref_trainer.condGANTrainer)
    t.my_dataset_flag = False
    t.summary_writer = _SummaryWriter()
    t.netG = ref_model.G_NET()
    t.netG.apply(ref_trainer.weights_init)
    nets = [ref_model.D_NET64, ref_model.D_NET128, ref_model.D_NET256][:cfg.BRANCH_NUM]
    t.netsD = [n() for n in nets]
    for n in t.netsD:
        n.apply(ref_trainer.weights_init)
    t.num_Ds = len(t.netsD)
    t.optimizerG, t.optimizersD = ref_trainer.define_optimizers(t.netG, t.netsD)
    t.criterion = nn.BCELoss()
    t.real_labels = torch.ones(batch_size)
    t.fake_labels = torch.zeros(batch_size)
    t.batch_size = batch_size
    return t, ref_model, ref_trainer


class ReferenceStepper:
    """The reference's own inner train loop (trainer.py:537-572 minus Inception) on the UNMODIFIED reference modules and
    the unmodified condGANTrainer.prepare_data / train_Dnet / train_Gnet, on the CPU: what `bench.py --impl reference`
    times when a reference tree is available (else it times the oracle port)."""

    def __init__(self, cfg, batch_size):
        import torch
        self.torch = torch
        self.t, self.ref_model, self.ref_trainer = build_reference_trainer(cfg, batch_size)
        self.avg_param_G = self.ref_trainer.copy_G_params(self.t.netG)
        self.count = 0

    def step(self, b):
        torch, t = self.torch, self.t
        data = (b["real"], b["wrong"], b["emb"], None, torch.as_tensor(b["labels"]))
        t.imgs_tcpu, t.real_imgs, t.wrong_imgs, t.txt_embedding, t.class_labels = t.prepare_data(data)
        t.fake_imgs, t.mu, t.logvar = t.netG(b["z"].clone().requires_grad_(True), t.txt_embedding)
        errD = [float(t.train_Dnet(i, self.count)) for i in range(t.num_Ds)]
        kl, err_g = t.train_Gnet(self.count)
        for p, avg_p in zip(t.netG.parameters(), self.avg_param_G):
            avg_p.mul_(0.999).add_(p.data, alpha=0.001)
        self.count += 1
        return errD, float(err_g), float(kl)
