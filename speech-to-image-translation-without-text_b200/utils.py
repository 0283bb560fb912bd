"""Host-side helpers shared by bench.py, the tests and user code."""
import torch
import torch.nn as nn


def _orthogonal_(w):
    """nn.init.orthogonal_ needs a view-compatible tensor; a FlatBucket exposes conv weights as permuted (OHWI-stored)
    views, so initialise a contiguous copy and write it through."""
    if w.is_contiguous():
        nn.init.orthogonal_(w, 1.0)
    else:
        w.copy_(nn.init.orthogonal_(torch.empty(w.shape, device=w.device, dtype=w.dtype), 1.0))


def weights_init(m):
    """Same initialisation the reference applies with net.apply(weights_init) (trainer.py:65-75):
    orthogonal (gain 1) for Conv / Linear weights, BN weight ~ N(1, 0.02), BN / Linear bias 0."""
    name = m.__class__.__name__
    if name.find("Conv") != -1:
        _orthogonal_(m.weight.data)
        invalidate_packs(m)
    elif name.find("BatchNorm") != -1:
        m.weight.data.normal_(1.0, 0.02)
        m.bias.data.fill_(0)
    elif name.find("Linear") != -1:
        _orthogonal_(m.weight.data)
        if m.bias is not None:
            m.bias.data.fill_(0.0)


def invalidate_packs(module):
    """Writes through `p.data` bump no version counter: tell the kernels' operand caches (bf16 packs, the FlatBucket
    mirror) that every parameter of `module` may have changed."""
    for p in module.parameters():
        p._sg2_version = getattr(p, "_sg2_version", 0) + 1
        p._sg2_mirror_stale = True


def load_params(model, new_param):
    """The reference's load_params (trainer.py:78-80: `p.data.copy_(new_p)`, used for the EMA swap around snapshot
    images and in save_model) plus the cache invalidation its `.data` writes cannot trigger."""
    for p, new_p in zip(model.parameters(), new_param):
        p.data.copy_(new_p)
    invalidate_packs(model)


def build_networks(cfg, device="cuda"):
    """G_NET + the BRANCH_NUM discriminators, initialised like trainer.load_network (trainer.py:162-184) does."""
    from . import model
    netG = model.G_NET().to(device)
    netG.apply(weights_init)
    netsD = [cls().to(device) for cls in (model.D_NET64, model.D_NET128, model.D_NET256)[:cfg.TREE.BRANCH_NUM]]
    for d in netsD:
        d.apply(weights_init)
    return netG, netsD


class _TrainerPatch:
    """sys.meta_path finder: lets the normal machinery load the reference's `trainer` module, then replaces its
    load_params with ours (same behaviour + operand-cache invalidation)."""

    def find_spec(self, name, path=None, target=None):
        if name != "trainer":
            return None
        import importlib.machinery
        import sys
        spec = importlib.machinery.PathFinder.find_spec(name, path or sys.path)
        if spec is None or spec.loader is None:
            return None
        inner = spec.loader.exec_module

        def exec_module(module):
            inner(module)
            patch_reference_trainer(module)

        spec.loader.exec_module = exec_module
        return spec


def patch_reference_trainer(trainer_module):
    if hasattr(trainer_module, "load_params"):
        trainer_module.load_params = load_params
    return trainer_module


def install_as_reference_model(inception=False):
    """Make `from model import G_NET, D_NET64, ...` (trainer.py:24) resolve to sg2b200.model, so the reference's
    unmodified main.py / trainer.py run on the CUDA kernels: call before importing the reference's trainer.
    Also binds the reference's global cfg (miscc.config.cfg) and arranges for the reference trainer's load_params
    (writes through `.data`) to invalidate the kernels' operand caches.
    inception=True: the aliased module is a proxy of sg2b200.model whose INCEPTION_V3 is the native scorer
    (sg2b200.inception), so the trainer's in-loop scoring (trainer.py:563-565) runs on these kernels too;
    sg2b200.model.INCEPTION_V3 itself is unchanged."""
    import sys
    import types
    from . import config, model
    if inception:
        from . import inception as inc
        proxy = types.ModuleType("model", model.__doc__)
        proxy.__dict__.update({k: v for k, v in vars(model).items() if not k.startswith("__")})
        proxy.INCEPTION_V3 = inc.INCEPTION_V3
        sys.modules["model"] = proxy
    else:
        sys.modules["model"] = model
    config.bind_reference_cfg()
    if "trainer" in sys.modules:
        patch_reference_trainer(sys.modules["trainer"])
    elif not any(isinstance(f, _TrainerPatch) for f in sys.meta_path):
        sys.meta_path.insert(0, _TrainerPatch())
    return model


def synthetic_batch(cfg, batch, seed, device="cpu", pin=False, n_classes=200):
    """Synthetic inputs of the benchmark (SURVEY.md section 8d): z, speech embedding, real / wrong image pyramids
    U(-1, 1) fp32 NCHW, class labels."""
    g = torch.Generator().manual_seed(seed)
    out = {"z": torch.randn(batch, cfg.GAN.Z_DIM, generator=g),
           "emb": torch.randn(batch, cfg.TEXT.DIMENSION, generator=g)}
    out["real"], out["wrong"] = [], []
    for i in range(cfg.TREE.BRANCH_NUM):
        s = 64 * 2 ** i
        out["real"].append(torch.rand(batch, 3, s, s, generator=g) * 2 - 1)
        out["wrong"].append(torch.rand(batch, 3, s, s, generator=g) * 2 - 1)
    lab = torch.randint(0, n_classes, (batch,), generator=g, dtype=torch.int32)
    if batch > 1:
        lab[1] = lab[0]          # at least one same-class pair so the class-aware loss is active
    out["labels"] = lab

    def mv(t):
        if pin:
            t = t.pin_memory()
        return t.to(device) if device != "cpu" else t
    return {k: ([mv(t) for t in v] if isinstance(v, list) else mv(v)) for k, v in out.items()}
