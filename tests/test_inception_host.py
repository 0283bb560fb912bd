"""CPU checks of the Inception-v3 scorer's host side: the state dict contract against torchvision, the BatchNorm folding,
the layer plan and its MMA row-utilisation report, the snapshot metrics in closed form, weight lookup without any
network access, and the reference-model install flag."""
import importlib.util
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F


def test_state_dict_matches_torchvision_and_loads_strictly():
    torchvision = pytest.importorskip("torchvision")
    from sg2b200 import inception
    tv = torchvision.models.inception_v3(weights=None, aux_logits=True, init_weights=False)
    ours = inception.INCEPTION_V3(random_init=True)
    a, b = ours.state_dict(), tv.state_dict()
    assert list(a) == ["model." + k for k in b]                      # the reference wraps torchvision as `self.model`
    assert all(a["model." + k].shape == v.shape for k, v in b.items())
    ours.model.load_state_dict(b)
    assert not ours.training and not any(p.requires_grad for p in ours.parameters())


def test_bn_folding_equals_conv_bn_relu_in_float64():
    from sg2b200 import inception
    torch.manual_seed(0)
    net = inception.Inception3()
    for name, m in net.named_modules():
        if not isinstance(m, inception.BasicConv2d):
            continue
        cin, cout, kh, kw, st, ph, pw = m.geo
        m.bn.running_mean.normal_()
        m.bn.running_var.uniform_(0.2, 3.0)
        m.bn.weight.data.normal_()
        m.bn.bias.data.normal_()
        x = torch.randn(1, cin, 9, 9, dtype=torch.float64)
        bn = m.bn.double().eval()
        ref = F.relu(bn(F.conv2d(x, m.conv.weight.double(), stride=st, padding=(ph, pw))))
        w, b = inception.fold_bn(m.conv.weight, m.bn.weight, m.bn.bias, m.bn.running_mean, m.bn.running_var, m.bn.eps)
        got = F.relu(F.conv2d(x, w, b, stride=st, padding=(ph, pw)))
        assert torch.allclose(got, ref, rtol=1e-10, atol=1e-10), name


def test_layer_plan_and_row_utilisation_report():
    from sg2b200 import inception
    plan = inception.layer_plan()
    assert len(plan) == 94
    assert abs(sum(L["macs"] for L in plan) / 1e9 - 5.711) < 5e-4
    pytest.importorskip("ctypes")
    import __graft_entry__
    __graft_entry__.build()
    rep = inception.utilisation_report(48)
    assert [r["name"] for r in rep] == [L["name"] for L in plan]
    for r in rep:
        assert r["useful_rows"] == 48 * r["Ho"] * r["Wo"] and r["issued_rows"] % 128 == 0
        assert 0.7 < r["row_use"] <= 1.0 and 0.6 <= r["col_use"] <= 1.0
    issued = sum(r["issued_rows"] * r["issued_cols"] * r["cin"] * r["kh"] * r["kw"] for r in rep)
    assert issued / (48 * sum(L["macs"] for L in plan)) < 1.3


def test_inception_score_closed_forms():
    from sg2b200 import metrics
    same = np.tile(np.array([[0.2, 0.3, 0.5]]), (6, 1))
    assert metrics.inception_score(same, 1)[0] == pytest.approx(1.0)
    n = 10
    p = np.full((n, n), 1e-9)
    np.fill_diagonal(p, 1.0)
    p /= p.sum(1, keepdims=True)
    assert metrics.inception_score(p, 1)[0] == pytest.approx(n, rel=1e-5)
    m, s = metrics.inception_score(np.concatenate([p, p]), 2)
    assert m == pytest.approx(n, rel=1e-5) and s == pytest.approx(0.0, abs=1e-6)
    nlpp = metrics.negative_log_posterior_probability(same, 2)
    assert nlpp[0] == pytest.approx(-np.log(0.5)) and nlpp[1] == pytest.approx(0.0)


def test_frechet_distance_closed_forms():
    from sg2b200 import metrics
    rng = np.random.default_rng(0)
    x = rng.standard_normal((400, 6))
    assert abs(metrics.frechet_distance(x, x)) < 1e-6
    # two Gaussians whose sample moments are exactly mu_a, diag(a) and mu_b, diag(b): FID = |mu_a - mu_b|^2 +
    # sum (a + b - 2 sqrt(a b))
    z = rng.standard_normal((2000, 4))
    z = (z - z.mean(0)) @ np.linalg.inv(np.linalg.cholesky(np.cov(z, rowvar=False))).T
    va, vb = np.array([1.0, 2.0, 0.5, 3.0]), np.array([2.0, 0.5, 0.5, 1.0])
    ma, mb = np.array([0.0, 1.0, -1.0, 2.0]), np.array([1.0, 1.0, 0.0, 0.0])
    a, b = z * np.sqrt(va) + ma, z * np.sqrt(vb) + mb
    ref = np.sum((ma - mb) ** 2) + np.sum(va + vb - 2 * np.sqrt(va * vb))
    assert metrics.frechet_distance(a, b) == pytest.approx(ref, rel=1e-8)


def _reference_trainer():
    ref = os.environ.get("SG2_REF")
    path = ref and os.path.join(ref, "StackGAN_v2", "trainer.py")
    if not path or not os.path.exists(path):
        pytest.skip("SG2_REF (reference checkout) not set")
    return path


def test_metrics_equal_the_reference_functions():
    path = _reference_trainer()
    from sg2b200 import metrics
    src = open(path).read()
    ns = {"np": np, "linalg": __import__("scipy.linalg", fromlist=["linalg"])}
    import ast
    tree = ast.parse(src)
    want = {"compute_inception_score", "negative_log_posterior_probability", "compute_frechet_distance"}
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in want:
            exec(compile(ast.Module([node], []), path, "exec"), ns)
    rng = np.random.default_rng(1)
    p = rng.dirichlet(np.ones(20), 40)
    if "compute_inception_score" in ns:
        assert np.allclose(ns["compute_inception_score"](p, 4), metrics.inception_score(p, 4))
    if "negative_log_posterior_probability" in ns:
        assert np.allclose(ns["negative_log_posterior_probability"](p, 4),
                           metrics.negative_log_posterior_probability(p, 4))


def test_missing_weights_raise_without_network(monkeypatch, tmp_path):
    from sg2b200 import inception

    def no_net(*a, **k):
        raise AssertionError("network access attempted")
    monkeypatch.setattr(socket.socket, "connect", no_net)
    monkeypatch.setattr(torch.hub, "load_state_dict_from_url", no_net)
    monkeypatch.setattr(torch.hub, "get_dir", lambda: str(tmp_path / "hub"))
    monkeypatch.setenv("SG2_INCEPTION_WEIGHTS", str(tmp_path / "none.pth"))
    with pytest.raises(FileNotFoundError) as e:
        inception.INCEPTION_V3()
    assert "none.pth" in str(e.value) and inception.WEIGHTS_FILE in str(e.value)
    with pytest.raises(FileNotFoundError):
        inception.INCEPTION_V3(weights=str(tmp_path / "other.pth"))


def test_weights_load_from_the_hub_cache_path(monkeypatch, tmp_path):
    from sg2b200 import inception
    src = inception.INCEPTION_V3(random_init=True)
    os.makedirs(tmp_path / "hub" / "checkpoints")
    torch.save(src.model.state_dict(), tmp_path / "hub" / "checkpoints" / inception.WEIGHTS_FILE)
    monkeypatch.setattr(torch.hub, "get_dir", lambda: str(tmp_path / "hub"))
    monkeypatch.delenv("SG2_INCEPTION_WEIGHTS", raising=False)
    m = inception.INCEPTION_V3()
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), src.state_dict().values()))


def test_install_flag_swaps_only_the_inception_alias(monkeypatch):
    from sg2b200 import inception, model, utils
    monkeypatch.delitem(sys.modules, "model", raising=False)
    utils.install_as_reference_model()
    assert sys.modules["model"] is model
    utils.install_as_reference_model(inception=True)
    alias = sys.modules["model"]
    assert alias is not model and alias.INCEPTION_V3 is inception.INCEPTION_V3
    for name in ("G_NET", "D_NET64", "D_NET128", "D_NET256", "D_NET512", "D_NET1024", "GLU"):
        assert getattr(alias, name) is getattr(model, name)
    with pytest.raises(NotImplementedError):
        model.INCEPTION_V3()
    monkeypatch.delitem(sys.modules, "model", raising=False)


def test_forward_rejects_cpu_tensors_and_train_mode():
    from sg2b200 import inception
    m = inception.INCEPTION_V3(random_init=True)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 64, 64))
    m.train()
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 64, 64))
