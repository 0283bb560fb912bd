"""CPU-side checks of the host logic: module/state-dict contract against the reference's golden state dicts,
weights_init dispatch, checkpoint round trip (incl. DataParallel 'module.' prefix), cfg binding."""
import io
import os

import numpy as np
import pytest
import torch

from oracle.stackgan_oracle import Cfg
from tests.parity_util import set_cfg

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_step_tiny.npz")
CFG_KEYS = sorted(["GF_DIM", "DF_DIM", "EMBEDDING_DIM", "Z_DIM", "R_NUM", "TEXT_DIM", "BRANCH_NUM"])


def _golden_cfg():
    z = np.load(GOLDEN)
    return z, Cfg(**{k: int(v) for k, v in zip(CFG_KEYS, z["meta_cfg"])})


def test_state_dict_matches_reference_names_shapes_and_order():
    from sg2b200 import model
    z, c = _golden_cfg()
    set_cfg(c)
    try:
        g = model.G_NET()
        ref = [k[3:] for k in z.files if k.startswith("g0/")]
        sd = g.state_dict()
        assert list(sd.keys()) == ref
        assert all(tuple(sd[k].shape) == z["g0/" + k].shape for k in ref)
        # parameters() ORDER drives Adam and the EMA zip (trainer.py:78-85, 240-251)
        assert [n for n, _ in g.named_parameters()] == [k for k in ref if "running" not in k and "num_batches" not in k]
        for i, cls in enumerate((model.D_NET64, model.D_NET128, model.D_NET256)):
            d = cls()
            ref = [k[5:] for k in z.files if k.startswith(f"d{i}_0/")]
            assert list(d.state_dict().keys()) == ref
            assert all(tuple(d.state_dict()[k].shape) == z[f"d{i}_0/" + k].shape for k in ref)
            # reference checkpoints load (strict), also with the DataParallel prefix (trainer.py:257)
            d.load_state_dict({k: torch.from_numpy(z[f"d{i}_0/" + k]) for k in ref})
            torch.nn.DataParallel(d).load_state_dict({"module." + k: torch.from_numpy(z[f"d{i}_0/" + k]) for k in ref})
    finally:
        set_cfg(Cfg())


def test_full_size_parameter_counts():
    """SURVEY.md section 5: G 21 239 696; D64 5 723 906; D128 18 834 178; D256 71 269 122 parameters."""
    from sg2b200 import model
    set_cfg(Cfg())
    counts = [sum(p.numel() for p in m().parameters()) for m in (model.G_NET, model.D_NET64, model.D_NET128, model.D_NET256)]
    assert counts == [21239696, 5723906, 18834178, 71269122]
    assert len(model.G_NET().state_dict()) == 107 and len(model.D_NET256().state_dict()) == 53


def test_weights_init_dispatch_and_checkpoint_roundtrip():
    from sg2b200 import model, utils
    set_cfg(Cfg(GF_DIM=8, DF_DIM=8, BRANCH_NUM=2))
    try:
        torch.manual_seed(0)
        g = model.G_NET()
        g.apply(utils.weights_init)
        w = g.h_net1.upsample1[1].weight.detach().reshape(g.h_net1.upsample1[1].weight.shape[0], -1)
        assert torch.allclose(w @ w.t(), torch.eye(w.shape[0]), atol=1e-4)            # orthogonal rows
        assert abs(float(g.h_net1.upsample1[2].weight.mean()) - 1.0) < 0.05 and float(g.h_net1.upsample1[2].bias.abs().max()) == 0
        buf = io.BytesIO()
        torch.save(g.state_dict(), buf)
        buf.seek(0)
        g2 = model.G_NET()
        g2.load_state_dict(torch.load(buf))
        assert all(torch.equal(a, b) for a, b in zip(g.state_dict().values(), g2.state_dict().values()))
    finally:
        set_cfg(Cfg())


def test_out_of_scope_classes_fail_loudly():
    from sg2b200 import model
    for cls in (model.D_NET512, model.D_NET1024, model.INCEPTION_V3):
        with pytest.raises(NotImplementedError):
            cls()


def test_modules_reject_cpu_inputs():
    from sg2b200 import model
    set_cfg(Cfg(BRANCH_NUM=1))
    try:
        with pytest.raises(RuntimeError):
            model.G_NET()(torch.randn(2, 100), torch.randn(2, 1024))
        with pytest.raises(RuntimeError):
            model.D_NET64()(torch.randn(2, 3, 64, 64), torch.randn(2, 128))
    finally:
        set_cfg(Cfg())


def test_split_k_factor_fills_whole_waves():
    """ops._auto_split (host logic, no kernel call): one CTA per (tile, split, parity group) on 148 SMs; the factor must
    not spill a few CTAs into an extra wave (D256's 1024->2048 layer at 3B = 72 tiles: 2 x 72 = 144, not 3 x 72 = 216),
    must count the output-parity groups of fused-upsample / stride-2-dgrad launches, and leaves full launches alone."""
    from sg2b200 import ops
    n_sm = ops.N_SM
    split = lambda *a, **k: ops._auto_split(*a, cap=32, **k)    # the wave logic, without the cluster-size cap
    assert split(72 * 16, 2048, 256) == 2            # 9 x 8 tiles
    assert split(24 * 16, 2048, 256) == 6            # 3 x 8 tiles
    assert split(24 * 16, 1024, 64, groups=4) == 3   # 3 x 4 tiles x 4 parity groups
    assert split(72 * 64 * 64, 256, 32) == 1         # thousands of tiles
    assert split(24 * 16, 512, 4) == 1               # too little K to split
    if ops.CLUSTER_SPLITK >= 2:                      # default: the splits of a tile form one cluster of at most this size
        assert ops._auto_split(24 * 16, 2048, 256) == min(6, ops.CLUSTER_SPLITK)
    for rows in (96, 384, 1152, 1536, 4608):
        for n in (256, 512, 1024, 2048):
            for kb in (16, 64, 144, 256, 288):
                for groups in (1, 4):
                    s = split(rows, n, kb, groups)
                    tiles = -(-rows // 128) * (n // 256) * groups
                    assert 1 <= s <= max(1, kb // 8)
                    if s > 1:   # a split launch is a whole number of (nearly) full waves, or a single partial one
                        waves = -(-tiles * s // n_sm)
                        assert tiles * s > (waves - 1) * n_sm + n_sm // 2 or waves == 1, (rows, n, kb, groups, s)


def test_bench_dump_outputs_fixed_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: flattened float32 / float64 arrays; a large one is reduced to a sample at positions that
    depend on its size only, so that two runs (or two builds) can be compared element for element."""
    import bench
    monkeypatch.setattr(bench, "DUMP_CAP", 100)
    x = torch.randn(7, 50)
    arrays = {"big": x, "small": torch.arange(6, dtype=torch.float64), "half": torch.ones(4, dtype=torch.bfloat16)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in arrays}
    assert a["big"].dtype == np.float32 and a["big"].shape == (100,) and len(np.unique(a["big"])) == 100
    assert np.isin(a["big"], x.numpy()).all()
    assert a["small"].dtype == np.float64 and np.array_equal(a["small"], np.arange(6))
    assert a["half"].dtype == np.float32 and np.array_equal(a["half"], np.ones(4, np.float32))
    assert all(np.array_equal(a[n], np.load(tmp_path / "b" / f"{n}.npy")) for n in arrays)
