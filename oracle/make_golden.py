"""ORACLE support — generate tests/golden/ref_step_tiny.npz by running the UNMODIFIED reference
(condGANTrainer.prepare_data / train_Dnet / train_Gnet + EMA, reference G_NET / D_NET*) on CPU in fp32.

    SG2_REF=<checkout>/StackGAN_v2 python oracle/make_golden.py     # needs a checkout of the reference

The fixture pins oracle/stackgan_oracle.py (tests/test_oracle.py): identical weights + inputs must give the
reference's losses, logits, images, gradients, BN running statistics and 4-step loss curve.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import golden, ref_loader  # noqa: E402
from oracle.stackgan_oracle import Cfg, synthetic_batch  # noqa: E402

TINY = dict(GF_DIM=4, DF_DIM=2, EMBEDDING_DIM=8, Z_DIM=10, R_NUM=2, TEXT_DIM=24, BRANCH_NUM=3)
BATCH = 3
STEPS = 4
EPS_SEED = 4242


def pooled(img, k=16):
    return torch.nn.functional.adaptive_avg_pool2d(img, k)


def run_reference(cfg, batch_size, steps):
    torch.manual_seed(99)
    t, ref_model, ref_trainer = ref_loader.build_reference_trainer(cfg, batch_size)
    init = {"g": {k: v.clone() for k, v in t.netG.state_dict().items()},
            "d": [{k: v.clone() for k, v in n.state_dict().items()} for n in t.netsD]}
    avg_param_G = ref_trainer.copy_G_params(t.netG)
    rec = {"steps": []}
    for s in range(steps):
        b = synthetic_batch(cfg, batch_size, seed=1234 + s)
        data = (b["real"], b["wrong"], b["emb"], None, torch.tensor(b["labels"]))
        t.imgs_tcpu, t.real_imgs, t.wrong_imgs, t.txt_embedding, t.class_labels = t.prepare_data(data)
        torch.manual_seed(EPS_SEED + s)        # the first draw after this is CA_NET's eps (model.py:190-193)
        t.fake_imgs, t.mu, t.logvar = t.netG(b["z"].clone().requires_grad_(True), t.txt_embedding)
        st = {"errD": [], "grads_d": []}
        for i in range(t.num_Ds):
            st["errD"].append(float(t.train_Dnet(i, s)))
            st["grads_d"].append({k: p.grad.detach().clone() for k, p in t.netsD[i].named_parameters()})
        kl, err_g = t.train_Gnet(s)
        st["kl"], st["errG_total"] = float(kl), float(err_g)
        st["grads_g"] = {k: p.grad.detach().clone() for k, p in t.netG.named_parameters()}
        for p, avg_p in zip(t.netG.parameters(), avg_param_G):
            avg_p.mul_(0.999).add_(p.data, alpha=0.001)
        st["fake"] = [f.detach().clone() for f in t.fake_imgs]
        st["mu"], st["logvar"] = t.mu.detach().clone(), t.logvar.detach().clone()
        rec["steps"].append(st)
    rec["final_g"] = {k: v.clone() for k, v in t.netG.state_dict().items()}
    rec["final_d"] = [{k: v.clone() for k, v in n.state_dict().items()} for n in t.netsD]
    rec["avg_g"] = [a.clone() for a in avg_param_G]
    return init, rec


def main():
    if not ref_loader.reference_available():
        raise SystemExit("no reference checkout found (set SG2_REF to its StackGAN_v2 directory)")
    cfg = Cfg(**TINY)
    init, rec = run_reference(cfg, BATCH, STEPS)
    out = {"meta_cfg": np.array([TINY[k] for k in sorted(TINY)], dtype=np.int64),
           "meta_batch_steps_seed": np.array([BATCH, STEPS, EPS_SEED], dtype=np.int64)}
    for k, v in init["g"].items():
        out["g0/" + k] = v.numpy()
    for i, sd in enumerate(init["d"]):
        for k, v in sd.items():
            out[f"d{i}_0/" + k] = v.numpy()
    s0 = rec["steps"][0]
    for i, f in enumerate(s0["fake"]):
        out[f"s0/fake{i}_pool16"] = pooled(f).numpy()
        out[f"s0/fake{i}_absmean"] = f.abs().mean().numpy()
    out["s0/fake0_full"] = s0["fake"][0].numpy()
    out["s0/mu"], out["s0/logvar"] = s0["mu"].numpy(), s0["logvar"].numpy()
    for k, v in s0["grads_g"].items():
        out["s0/grad_g/" + k] = v.numpy()
    for i, gd in enumerate(s0["grads_d"]):
        for k, v in gd.items():
            out[f"s0/grad_d{i}/" + k] = v.numpy()
    out["curve_errD"] = np.array([st["errD"] for st in rec["steps"]], dtype=np.float64)
    out["curve_errG"] = np.array([st["errG_total"] for st in rec["steps"]], dtype=np.float64)
    out["curve_kl"] = np.array([st["kl"] for st in rec["steps"]], dtype=np.float64)
    # end state after STEPS steps: every buffer (BN running stats, num_batches_tracked) and a norm per parameter
    for k, v in rec["final_g"].items():
        out["gN/" + k] = v.numpy() if "running" in k or "num_batches" in k else np.array(v.double().norm().item())
    for i, sd in enumerate(rec["final_d"]):
        for k, v in sd.items():
            out[f"d{i}_N/" + k] = v.numpy() if "running" in k or "num_batches" in k else np.array(v.double().norm().item())
    out["avg_g_norms"] = np.array([a.double().norm().item() for a in rec["avg_g"]])
    out = golden.shrink(out)
    path = os.path.join(ROOT, "tests", "golden", "ref_step_tiny.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", "errD", out["curve_errD"][0], "errG", out["curve_errG"][0])


if __name__ == "__main__":
    main()
