"""Pin the oracle (oracle/stackgan_oracle.py) to the reference: committed golden vectors produced by the
unmodified reference (oracle/make_golden.py), and — where a reference checkout is given (SG2_REF) — the reference
itself."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle.golden import sketch
from oracle.stackgan_oracle import Cfg, OracleTrainer, param_keys, synthetic_batch

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_step_tiny.npz")
CFG_KEYS = sorted(["GF_DIM", "DF_DIM", "EMBEDDING_DIM", "Z_DIM", "R_NUM", "TEXT_DIM", "BRANCH_NUM"])


def _load():
    z = np.load(GOLDEN)
    cfg = Cfg(**{k: int(v) for k, v in zip(CFG_KEYS, z["meta_cfg"])})
    batch, steps, eps_seed = (int(v) for v in z["meta_batch_steps_seed"])
    g0 = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("g0/")}
    ds = [{k[5:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(f"d{i}_0/")} for i in range(cfg.BRANCH_NUM)]
    return z, cfg, batch, steps, eps_seed, g0, ds


def _rel(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _rel_ref(z, a, key):
    """_rel against the reference array `key`, or, for the large ones the fixture keeps as a sketch, the same estimate
    from the sketches (oracle/golden.py)."""
    if key in z.files:
        return _rel(a, z[key])
    return _rel(sketch(a), z["sketch/" + key])


@pytest.fixture(scope="module")
def run():
    z, cfg, batch, steps, eps_seed, g0, ds = _load()
    tr = OracleTrainer(cfg, g0, ds)
    outs = []
    for s in range(steps):
        b = synthetic_batch(cfg, batch, seed=1234 + s)
        torch.manual_seed(eps_seed + s)
        b["eps"] = torch.FloatTensor(batch, cfg.EMBEDDING_DIM).normal_()   # the draw model.py:190-193 makes
        outs.append(tr.step(b, keep_grads=(s == 0)))
    return z, cfg, tr, outs


def test_state_dict_contract(run):
    """Key names, order and shapes equal the reference's state_dict (checkpoint drop-in)."""
    from oracle.stackgan_oracle import init_d_state, init_g_state
    z, cfg, tr, _ = run
    ref_keys = [k[3:] for k in z.files if k.startswith("g0/")]
    mine = init_g_state(cfg)
    assert list(mine.keys()) == ref_keys
    for k in ref_keys:
        assert tuple(mine[k].shape) == z["g0/" + k].shape, k
    for i in range(cfg.BRANCH_NUM):
        ref_keys = [k[5:] for k in z.files if k.startswith(f"d{i}_0/")]
        mine = init_d_state(cfg, i)
        assert list(mine.keys()) == ref_keys, i
        for k in ref_keys:
            assert tuple(mine[k].shape) == z[f"d{i}_0/" + k].shape, (i, k)


def test_forward_matches_reference(run):
    z, cfg, tr, outs = run
    o = outs[0]
    assert _rel_ref(z, o["fake"][0], "s0/fake0_full") < 1e-5
    for i in range(cfg.BRANCH_NUM):
        pooled = torch.nn.functional.adaptive_avg_pool2d(o["fake"][i], 16)
        assert _rel(pooled, z[f"s0/fake{i}_pool16"]) < 1e-5
        assert abs(float(o["fake"][i].abs().mean()) - float(z[f"s0/fake{i}_absmean"])) < 1e-6
    assert _rel(o["mu"], z["s0/mu"]) < 1e-6
    assert _rel(o["logvar"], z["s0/logvar"]) < 1e-6


def test_losses_track_reference_curve(run):
    z, cfg, tr, outs = run
    errD = np.array([[float(e) for e in o["errD"]] for o in outs])
    errG = np.array([float(o["errG_total"]) for o in outs])
    kl = np.array([float(o["kl"]) for o in outs])
    np.testing.assert_allclose(errD, z["curve_errD"], rtol=2e-4)
    np.testing.assert_allclose(errG, z["curve_errG"], rtol=2e-4)
    np.testing.assert_allclose(kl, z["curve_kl"], rtol=2e-4)


def test_gradients_match_reference(run):
    z, cfg, tr, outs = run
    o = outs[0]
    worst = 0.0
    for k, g in o["grads_g"].items():
        worst = max(worst, _rel_ref(z, g, "s0/grad_g/" + k))
    for i, gd in enumerate(o["grads_d"]):
        for k, g in gd.items():
            worst = max(worst, _rel_ref(z, g, f"s0/grad_d{i}/" + k))
    assert worst < 2e-4, worst


def test_end_state_matches_reference(run):
    """After 4 Adam steps: BN running stats, num_batches_tracked (G: +1/step, D: +4/step), parameter norms, EMA."""
    z, cfg, tr, outs = run
    for name, sd in [("gN/", tr.g)] + [(f"d{i}_N/", tr.ds[i]) for i in range(cfg.BRANCH_NUM)]:
        for k, v in sd.items():
            ref = z[name + k]
            if "num_batches" in k:
                assert int(v) == int(ref), (name, k)
            elif "running" in k:
                assert _rel(v, ref) < 1e-4, (name, k)
            else:
                assert abs(float(v.detach().double().norm()) - float(ref)) <= 2e-4 * max(1.0, float(ref)), (name, k)
    norms = np.array([float(a.double().norm()) for a in tr.avg_g])
    np.testing.assert_allclose(norms, z["avg_g_norms"], rtol=1e-4, atol=1e-8)


def test_direct_against_reference_modules():
    """The oracle's module forwards alone (g_forward, d_forward; no trainer, no optimiser) on the reference's initial
    weights and step-0 batch, against what the reference's own G_NET and D_NET256 produced there: the three images, mu
    and logvar, and D_NET256's train_Dnet loss (trainer.py:375-427) with the gradient of every D_NET256 weight, which
    depend on each of its logits and, through backward, on every activation including x_immediate."""
    from oracle.stackgan_oracle import bce, d_forward, g_forward
    z, cfg, batch, _, eps_seed, g0, ds = _load()
    b = synthetic_batch(cfg, batch, seed=1234)
    torch.manual_seed(eps_seed)
    eps = torch.FloatTensor(batch, cfg.EMBEDDING_DIM).normal_()          # the draw model.py:190-193 makes
    fake, mu, logvar = g_forward({k: v.clone() for k, v in g0.items()}, b["z"], b["emb"], eps, cfg, True)
    assert _rel_ref(z, fake[0], "s0/fake0_full") < 1e-5
    for i, f in enumerate(fake):
        assert _rel(torch.nn.functional.adaptive_avg_pool2d(f, 16), z[f"s0/fake{i}_pool16"]) < 1e-5
    assert _rel(mu, z["s0/mu"]) < 1e-6 and _rel(logvar, z["s0/logvar"]) < 1e-6
    which = cfg.BRANCH_NUM - 1                                            # D_NET256
    dsd = {k: v.clone() for k, v in ds[which].items()}
    keys = param_keys(dsd)
    for k in keys:
        dsd[k].requires_grad_(True)
    ones, zeros, u = torch.ones(batch), torch.zeros(batch), cfg.UNCOND_LOSS
    rl, _ = d_forward(dsd, b["real"][which], mu, which, cfg)
    wl, _ = d_forward(dsd, b["wrong"][which], mu, which, cfg)
    fl, _ = d_forward(dsd, fake[which].detach(), mu, which, cfg)
    err = (bce(rl[0], ones) + u * bce(rl[1], ones) + bce(wl[0], zeros) + u * bce(wl[1], ones)
           + bce(fl[0], zeros) + u * bce(fl[1], zeros))
    np.testing.assert_allclose(float(err.detach()), z["curve_errD"][0][which], rtol=2e-4)
    grads = torch.autograd.grad(err, [dsd[k] for k in keys])
    worst = max(_rel_ref(z, g, f"s0/grad_d{which}/" + k) for k, g in zip(keys, grads))
    assert worst < 2e-4, worst


@pytest.mark.skipif(not ref_loader.reference_available(), reason="needs a reference checkout (SG2_REF)")
def test_direct_against_live_reference_modules():
    """Same weights + inputs through the reference's own G_NET / D_NET256 (from a checkout) and through the oracle."""
    from oracle.stackgan_oracle import d_forward, g_forward
    cfg = Cfg(GF_DIM=8, DF_DIM=4, EMBEDDING_DIM=16, Z_DIM=12, R_NUM=2, TEXT_DIM=20, BRANCH_NUM=3)
    ref_model, ref_trainer, _ = ref_loader.load_reference(cfg)
    torch.manual_seed(5)
    netG = ref_model.G_NET()
    netG.apply(ref_trainer.weights_init)
    netD = ref_model.D_NET256()
    netD.apply(ref_trainer.weights_init)
    b = synthetic_batch(cfg, 2, seed=7)
    gsd = {k: v.clone() for k, v in netG.state_dict().items()}
    dsd = {k: v.clone() for k, v in netD.state_dict().items()}
    torch.manual_seed(11)
    fake, mu, logvar = netG(b["z"], b["emb"])
    torch.manual_seed(11)
    eps = torch.FloatTensor(2, cfg.EMBEDDING_DIM).normal_()
    ofake, omu, ologvar = g_forward(gsd, b["z"], b["emb"], eps, cfg, True)
    for a, r in zip(ofake, fake):
        assert _rel(a, r.detach()) < 1e-5
    assert _rel(omu, mu.detach()) < 1e-6
    logits, x_imm = netD(b["real"][2], mu.detach())
    ologits, ox = d_forward(dsd, b["real"][2], omu, 2, cfg, True)
    assert _rel(ox, x_imm.detach()) < 1e-5
    assert _rel(ologits[0], logits[0].detach()) < 1e-5 and _rel(ologits[1], logits[1].detach()) < 1e-5
    # BN running stats were updated identically
    for k, v in netG.state_dict().items():
        if "running" in k:
            assert _rel(gsd[k], v) < 1e-5, k
