"""GPU parity of the Inception-v3 scorer (sg2b200.inception): every convolution geometry of the network on the gather
kernel (bias + ReLU epilogue, channel slices in and out), the stem / pool / average / softmax kernels, and the whole
network against float64 torchvision with the ideal-bf16 yardstick of tests/test_gpu_nets.py."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

YARD = 1.3


def _rel(a, b):
    a, b = a.detach().double().flatten(), b.detach().double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _bf(t):
    return t.bfloat16().float()


def _record(name, value):
    """Measured values of this file, written to $SG2_RECORD_DIR/inception_parity.json when that is set."""
    out = os.environ.get("SG2_RECORD_DIR")
    if not out or not os.path.isdir(out):
        return
    path = os.path.join(out, "inception_parity.json")
    d = json.load(open(path)) if os.path.exists(path) else {}
    d[name] = value
    json.dump(d, open(path, "w"), indent=1)


@pytest.fixture(autouse=True)
def _strict():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


# --------------------------------------------------------------------------------------------- convolutions
GEOMETRIES = [  # B, H, Cin, Cout, kh, kw, stride, ph, pw: each row of the network's geometry table at real sizes
    (2, 73, 64, 80, 1, 1, 1, 0, 0), (4, 17, 768, 192, 1, 1, 1, 0, 0), (3, 8, 2048, 448, 1, 1, 1, 0, 0),
    (2, 35, 192, 48, 1, 1, 1, 0, 0),
    (2, 147, 32, 64, 3, 3, 1, 1, 1), (3, 35, 64, 96, 3, 3, 1, 1, 1), (3, 8, 448, 384, 3, 3, 1, 1, 1),
    (2, 149, 32, 32, 3, 3, 1, 0, 0), (2, 73, 80, 192, 3, 3, 1, 0, 0),
    (3, 17, 160, 160, 1, 7, 1, 0, 3), (3, 17, 128, 192, 7, 1, 1, 3, 0),
    (2, 35, 288, 384, 3, 3, 2, 0, 0), (3, 35, 96, 96, 3, 3, 2, 0, 0), (3, 17, 192, 320, 3, 3, 2, 0, 0),
    (2, 35, 48, 64, 5, 5, 1, 2, 2),
    (3, 8, 384, 384, 1, 3, 1, 0, 1), (3, 8, 384, 384, 3, 1, 1, 1, 0),
]


@pytest.mark.parametrize("B,H,Ci,Co,kh,kw,st,ph,pw", GEOMETRIES)
def test_conv2d_geometry_into_channel_slice(B, H, Ci, Co, kh, kw, st, ph, pw):
    """relu(conv + bias) from a channel slice of a wider input into a channel slice of a NaN-prefilled wider output:
    rel err <= 5e-3 against float64 conv2d on the same bf16 operands, and no byte outside the slice changes."""
    from sg2b200 import ops
    g = torch.Generator().manual_seed(H * 7 + Ci + Co + kh * 3 + st)
    xc0, Cx = 16, Ci + 48
    oc0, Cy = 64, Co + 96
    x = torch.randn(B, H, H, Cx, generator=g).bfloat16().cuda()
    w = (torch.randn(Co, kh, kw, Ci, generator=g) / (Ci * kh * kw) ** 0.5).bfloat16().cuda()
    b = (0.1 * torch.randn(Co, generator=g)).cuda()
    Ho, Wo = ops.conv2d_out_hw(H, H, kh, kw, st, ph, pw)
    y = torch.full((B, Ho, Wo, Cy), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.conv2d_fprop(x, Ci, w.reshape(Co, -1).contiguous(), b, y, Co, kh, kw, st, ph, pw, True, xc0, oc0)
    torch.cuda.synchronize()
    xin = x[..., xc0:xc0 + Ci].permute(0, 3, 1, 2).double()
    ref = F.relu(F.conv2d(xin, w.permute(0, 3, 1, 2).double(), b.double(), stride=st, padding=(ph, pw)))
    got = y[..., oc0:oc0 + Co].permute(0, 3, 1, 2)
    assert _rel(got, ref) <= 5e-3
    assert torch.isnan(y[..., :oc0].float()).all() and torch.isnan(y[..., oc0 + Co:].float()).all()


def test_conv2d_plan_covers_every_layer():
    from sg2b200 import inception
    rep = inception.utilisation_report(48)
    assert len(rep) == 94 and all(0.7 < r["row_use"] <= 1.0 for r in rep)


# --------------------------------------------------------------------------------------------- small kernels
def _stem_ref(img):
    x = img.double() * 0.5 + 0.5
    mean = torch.tensor([0.485, 0.456, 0.406], dtype=torch.float64, device=img.device).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225], dtype=torch.float64, device=img.device).view(1, 3, 1, 1)
    x = (x - mean) / std
    return F.interpolate(x, size=(299, 299), mode="bilinear", align_corners=False)


@pytest.mark.parametrize("S", [64, 256, 299, 400])
def test_inception_stem(S):
    from sg2b200 import ops
    g = torch.Generator().manual_seed(S)
    img = (torch.rand(2, 3, S, S, generator=g) * 2 - 1).cuda()
    col = ops.inception_stem(img).float()
    x = _stem_ref(img)
    ref = F.unfold(x, 3, stride=2)                                   # (B, 3*9 (c, ky, kx), 149*149)
    ref = ref.view(2, 3, 9, 149 * 149).permute(0, 3, 2, 1).reshape(2, 149, 149, 27)   # -> (ky, kx, c)
    assert _rel(col[..., :27], ref) <= 5e-3
    assert (col[..., 27:] == 0).all()


def test_pools_average_softmax():
    from sg2b200 import ops
    g = torch.Generator().manual_seed(3)
    x = torch.randn(3, 17, 17, 96, generator=g).bfloat16().cuda()
    xd = x.permute(0, 3, 1, 2).double()
    out = torch.full((3, 8, 8, 160), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.maxpool3s2(x, out, 32)
    assert torch.equal(out[..., 32:128].permute(0, 3, 1, 2).double(), F.max_pool2d(xd, 3, 2))
    assert torch.isnan(out[..., :32].float()).all() and torch.isnan(out[..., 128:].float()).all()
    avg = ops.avgpool3s1(x).permute(0, 3, 1, 2)
    assert _rel(avg, F.avg_pool2d(xd, 3, 1, 1, count_include_pad=True)) <= 5e-3
    y = torch.randn(4, 8, 8, 2048, generator=g).bfloat16().cuda()
    assert _rel(ops.global_avg(y), y.double().mean((1, 2))) <= 1e-5
    z = (3 * torch.randn(5, 1000, generator=g)).cuda()
    assert _rel(ops.softmax_rows(z), torch.softmax(z.double(), 1)) <= 1e-5


# --------------------------------------------------------------------------------------------- whole network
@pytest.fixture(scope="module")
def nets():
    """torchvision Inception3 with random weights and BatchNorm running statistics calibrated once (float64, train mode,
    momentum 1) so that activations keep their scale through the 94 layers; the scorer holds the same state dict."""
    torchvision = pytest.importorskip("torchvision")
    from sg2b200 import inception
    torch.manual_seed(0)
    tv = torchvision.models.inception_v3(weights=None, aux_logits=True, init_weights=True).cuda().double()
    for m in tv.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.momentum = 1.0
    tv.train()
    with torch.no_grad():
        tv(_stem_ref(torch.rand(16, 3, 128, 128, device="cuda") * 2 - 1))
    tv.eval()
    ours = inception.INCEPTION_V3(random_init=True)
    ours.model.load_state_dict(tv.state_dict())
    return tv, ours


def _tv_forward(tv, x, emulate):
    """torchvision's forward from the resized input; emulate: folded BN with bf16 weights, bf16 conv / pool outputs
    (ideal bf16 storage), else float64 as is. -> (softmax, pool3)."""
    from sg2b200 import inception
    hooks = []
    feats = {}
    if emulate:
        def conv_hook(m, inp, out):
            w, b = inception.fold_bn(m.conv.weight, m.bn.weight, m.bn.bias, m.bn.running_mean, m.bn.running_var, m.bn.eps)
            y = F.conv2d(_bf(inp[0].float()), _bf(w.float()), b.float(), m.conv.stride, m.conv.padding)
            return _bf(F.relu(y)).double()
        for m in tv.modules():
            if type(m).__name__ == "BasicConv2d":
                hooks.append(m.register_forward_hook(conv_hook))
    hooks.append(tv.avgpool.register_forward_hook(lambda m, i, o: feats.setdefault("pool3", o.flatten(1))))
    try:
        with torch.no_grad():
            logits = tv(x)
    finally:
        for h in hooks:
            h.remove()
    return torch.softmax(logits.double(), 1), feats["pool3"].double()


@pytest.mark.parametrize("B,S", [(8, 64), (48, 256)])
def test_whole_network_against_float64(nets, B, S):
    tv, ours = nets
    g = torch.Generator().manual_seed(B + S)
    img = (torch.rand(B, 3, S, S, generator=g) * 2 - 1).cuda()
    pred, pool3 = ours(img)
    x = _stem_ref(img)
    p64, f64 = _tv_forward(tv, x, False)
    pem, fem = _tv_forward(tv, x, True)
    e_pred, e_pool = _rel(pred, p64), _rel(pool3, f64)
    y_pred, y_pool = _rel(pem, p64), _rel(fem, f64)
    _record(f"whole_B{B}_S{S}", dict(pred=e_pred, pool3=e_pool, ideal_pred=y_pred, ideal_pool3=y_pool))
    print(f"B={B} S={S}: pred {e_pred:.3e} (ideal bf16 {y_pred:.3e}), pool3 {e_pool:.3e} (ideal bf16 {y_pool:.3e})")
    assert pred.dtype == torch.float32 and pool3.shape == (B, 2048) and not pred.requires_grad
    assert torch.allclose(pred.sum(1), torch.ones(B, device="cuda"), atol=1e-4)
    assert e_pred <= YARD * y_pred + 1e-4 and e_pool <= YARD * y_pool + 1e-4


def test_fid_of_native_features(nets):
    from sg2b200 import metrics
    tv, ours = nets
    g = torch.Generator().manual_seed(11)
    fn, f64, fem = [], [], []
    for _ in range(10):
        img = (torch.rand(50, 3, 64, 64, generator=g) * 2 - 1).cuda()
        fn.append(ours(img)[1].double().cpu())
        x = _stem_ref(img)
        f64.append(_tv_forward(tv, x, False)[1].cpu())
        fem.append(_tv_forward(tv, x, True)[1].cpu())
    fn, f64, fem = (torch.cat(t).numpy() for t in (fn, f64, fem))
    d_ours, d_ideal = metrics.frechet_distance(fn, f64), metrics.frechet_distance(fem, f64)
    _record("fid_500", dict(native_vs_f64=d_ours, ideal_bf16_vs_f64=d_ideal))
    print(f"FID(native, f64) {d_ours:.4e}  FID(ideal bf16, f64) {d_ideal:.4e}")
    # floor: the round-off of the 2048 x 2048 matrix square root, relative to the features' total variance
    assert d_ours <= YARD * d_ideal + 1e-9 * float(np.trace(np.cov(f64, rowvar=False)))


def test_scorer_is_reproducible_and_refolds_on_load(nets):
    tv, ours = nets
    img = (torch.rand(6, 3, 128, 128) * 2 - 1).cuda()
    p1, f1 = ours(img)
    p2, f2 = ours(img)
    assert torch.equal(p1, p2) and torch.equal(f1, f2)
    sd = {k: v.clone() for k, v in ours.model.state_dict().items()}
    sd["fc.bias"] += 1.0
    sd["Mixed_7c.branch_pool.bn.bias"] += 0.5
    ours.model.load_state_dict(sd)
    try:
        p3, f3 = ours(img)
        assert not torch.equal(f1, f3) and not torch.equal(p1, p3)
    finally:
        ours.model.load_state_dict(tv.state_dict())
    p4, f4 = ours(img)
    assert torch.equal(p1, p4) and torch.equal(f1, f4)


def test_train_mode_and_cpu_inputs_are_rejected(nets):
    _, ours = nets
    with pytest.raises(RuntimeError):
        ours(torch.zeros(2, 3, 64, 64))
    ours.train()
    try:
        with pytest.raises(RuntimeError):
            ours(torch.zeros(2, 3, 64, 64, device="cuda"))
    finally:
        ours.eval()


# --------------------------------------------------------------------------------------------- captured train step
def test_captured_step_scores_without_touching_training_state(nets):
    """CapturedStep with and without the scorer from the same snapshot, same given noise, B = 24, 3 stages: every loss,
    parameter, Adam moment, EMA weight and BatchNorm buffer agrees after 3 replays (to the 2^-53 order dependence of the
    step's fp64 statistics atomics, as in test_gpu_captured.py), and the graph's scores equal standalone scorer calls on
    the last step's fake256 (recomputed eagerly from the restored snapshot) and on the real batch."""
    from sg2b200 import trainer
    from tests.parity_util import build_trainer_and_oracles, rel, snapshot_diff, train_batch
    _, scorer = nets
    B = 24
    cfg, _, _, _, tr, _ = build_trainer_and_oracles(3, seed=0, n_oracles=0)
    batches = [train_batch(cfg, B, 500 + s) for s in range(3)]
    snap0 = tr.snapshot()

    def load(cap, b):
        cap.load(b["emb"], b["real"], b["wrong"], b["labels"], z=b["z"], eps=b["eps"])

    def run(sc):
        tr.restore(snap0)
        cap = trainer.CapturedStep(tr, B, warmup=2, draw_noise=False, scorer=sc)
        load(cap, batches[0])
        cap.capture()
        tr.restore(snap0)
        ls = []
        for k, b in enumerate(batches):
            if k == len(batches) - 1:
                torch.cuda.synchronize()
                snap_last = tr.snapshot()
            load(cap, b)
            ls.append(cap.replay().clone())
        torch.cuda.synchronize()
        return cap, tr.snapshot(), torch.stack(ls), snap_last

    _, s_plain, l_plain, _ = run(None)
    cap, s_score, l_score, snap_last = run(scorer)
    d, bitwise = snapshot_diff(s_score, s_plain)
    _record("captured_step", dict(max_rel_state_diff=d, bitwise=bool(bitwise), losses_equal=bool(torch.equal(l_score, l_plain))))
    assert d <= 1e-6 and rel(l_score, l_plain) <= 1e-6, (d, bitwise)
    # the scores of the last replay: eager recomputation of that step's fake256 from the snapshot before it
    tr.restore(snap_last)
    b = batches[-1]
    last = {}
    tr.step(b["z"], b["emb"], b["real"], b["wrong"], b["labels"], eps=b["eps"],
            on_img=lambda i, img: last.__setitem__(i, img.clone()))
    pf, ff = scorer(last[2])
    pr, fr = scorer(b["real"][-1])
    torch.cuda.synchronize()
    assert rel(cap.pool3_fake, ff) <= 1e-6 and rel(cap.pred_fake, pf) <= 1e-6
    assert torch.equal(cap.pool3_real, fr) and torch.equal(cap.pred_real, pr)
