"""Every convolution and linear call of one production train step, and of the Inception scorer, checked per element
against float64 at the moment it is made (tests/launch_ref.py: references on the packed operands, bounds derived from
where the kernels round). These are the shapes, split-K factors, statistics groups and kernel variants the unit tests of
tests/test_gpu_kernels.py never reach: 72-row discriminator passes, _auto_split factors, production pixel counts,
the data-parallel grids (8 SMs reserved, CTA-pair kernels off) and the fp32-accurate mode."""
import time

import pytest
import torch

from tests import launch_ref as L
from tests.parity_util import build_trainer_and_oracles, train_batch

pytestmark = pytest.mark.gpu


def _step_rows(branches, B, precision="bf16", data_parallel=False, keep=None):
    """Two warm-up steps (weights off their initial values), then one eager step inside the checker."""
    from sg2b200 import _lib, config
    config.set_precision(precision)
    try:
        if data_parallel:
            _lib.call("sg2_set_sm_reserve", 8)
            _lib.call("sg2_set_pair_kernels", 0)
        cfg, _, _, _, tr, _ = build_trainer_and_oracles(branches, seed=0, n_oracles=0)
        assert tr.precise == (precision == "fp32")
        for s in range(2):
            b = train_batch(cfg, B, 100 + s)
            tr.step(b["z"], b["emb"], b["real"], b["wrong"], b["labels"], eps=b["eps"])
        torch.cuda.synchronize()
        b = train_batch(cfg, B, 200)
        t0 = time.time()
        with L.checked(keep) as chk:
            losses = tr.step(b["z"], b["emb"], b["real"], b["wrong"], b["labels"], eps=b["eps"])
        torch.cuda.synchronize()
        chk.seconds = time.time() - t0
        assert bool(torch.isfinite(losses).all())
        return chk
    finally:
        if data_parallel:
            _lib.call("sg2_set_sm_reserve", 0)
            _lib.call("sg2_set_pair_kernels", -1)
        config.set_precision("bf16")


def _assert_all_checked(name, chk, ops_expected):
    print(f"\n{name}: {chk.calls} calls checked in {chk.seconds:.1f} s\n" + chk.table())
    L.record(name, {"calls": chk.calls, "seconds": round(chk.seconds, 2), "worst": chk.worst_by_kind(),
                    "rows": chk.rows})
    assert chk.unchecked == [], chk.unchecked
    assert chk.calls == len(chk.rows) > 0
    assert {r["op"] for r in chk.rows} >= set(ops_expected)
    bad = [r for r in chk.rows if not r["ratio"] <= 1.0]
    assert not bad, "launches over their bound:\n" + "\n".join(str(r) for r in bad)


STEP_OPS = ("fprop", "dgrad", "wgrad", "linear_fwd", "linear_bwd_w", "linear_bwd_x")


def _keep(row):
    """Launches the fault-injection test re-checks: grouped statistics, 256^2 output maps, the largest contractions."""
    if row["op"] != "fprop":
        return False
    Ho = L.out_hw(getattr(L, row["kind"]), row["H"], row["W"])[0]
    return row["groups"] == 3 or Ho == 256 or L.k_fprop(getattr(L, row["kind"]), row["Cin"]) >= 9 * 1024


@pytest.fixture(scope="module")
def step_b24():
    return _step_rows(3, 24, keep=_keep)


def test_step_b24_every_launch(step_b24):
    _assert_all_checked("3stage_B24", step_b24, STEP_OPS)
    assert any(r["groups"] == 3 for r in step_b24.rows)          # the 72-row discriminator passes
    assert any("bias9" in r["epi"] for r in step_b24.rows)        # jointConv
    assert any("lrelu" in r["epi"] for r in step_b24.rows)        # D stems


def test_step_b64_every_launch():
    _assert_all_checked("3stage_B64", _step_rows(3, 64), STEP_OPS)


def test_step_b24_data_parallel_grids_every_launch():
    _assert_all_checked("3stage_B24_dp_grids", _step_rows(3, 24, data_parallel=True), STEP_OPS)


def test_step_fp32_accurate_every_launch():
    chk = _step_rows(3, 24, precision="fp32")
    _assert_all_checked("3stage_B24_fp32", chk, STEP_OPS)
    assert any(r["dtype"] == "float32" and r["groups"] == 3 for r in chk.rows)


@pytest.mark.parametrize("B,S", [(48, 256), (25, 64)])
def test_inception_scorer_every_launch(B, S):
    from sg2b200 import inception
    torch.manual_seed(0)
    net = inception.INCEPTION_V3(random_init=True).cuda()
    img = torch.rand(B, 3, S, S, generator=torch.Generator().manual_seed(B)).cuda() * 2 - 1
    t0 = time.time()
    with L.checked() as chk:
        pred, pool3 = net(img)
    torch.cuda.synchronize()
    chk.seconds = time.time() - t0
    assert bool(torch.isfinite(pred).all()) and bool(torch.isfinite(pool3).all())
    _assert_all_checked(f"inception_B{B}_S{S}", chk, ("conv2d", "linear_fwd"))
    assert sum(r["op"] == "conv2d" for r in chk.rows) == 94
    assert sum(r["op"] == "linear_fwd" for r in chk.rows) == 1


def test_checker_rejects_faults_in_real_launches(step_b24):
    """Seeded faults applied to real kernel outputs of the B = 24 step: the largest-K gather launch, a launch with a
    256^2 output map and a 72-row grouped-statistics launch."""
    kept = step_b24.kept
    assert kept
    by_k = max(kept, key=lambda rk: L.k_fprop(getattr(L, rk[0]["kind"]), rk[0]["Cin"]))
    big = next(rk for rk in kept if L.out_hw(getattr(L, rk[0]["kind"]), rk[0]["H"], rk[0]["W"])[0] == 256)
    grouped = next(rk for rk in kept if rk[0]["groups"] == 3 and rk[1]["stats_delta"] is not None)
    assert L.k_fprop(getattr(L, by_k[0]["kind"]), by_k[0]["Cin"]) == 9 * 2048
    for row, k in (by_k, big, grouped):
        kind = getattr(L, row["kind"])

        def chk(y):
            return L.check_fprop(kind, k["x"], k["wpk"], y, row["Cout"], k["splits"], k["act"], k["bias9"])

        assert chk(k["y"]) <= 1.0, row
        y = k["y"].clone()
        y[1, y.shape[1] // 2] = k["y"][0, y.shape[1] // 2]            # one output row from the neighbouring image
        assert chk(y) > 1.0, row
        y = k["y"].clone()
        y[0, 0, 1, 3] = k["y"][0, 0, 1, 3].float() * -1.5 + 0.25     # one element at a stale value
        assert chk(y) > 1.0, row
        if kind == L.CONV3 and k["act"] == 0 and k["bias9"] is None:
            # one border tap of one pixel dropped: pixel (0, 1), tap (2, 1) reads x[b, 1, 1]
            y = k["y"].double().clone()
            y[2, 0, 1] -= k["x"][2, 1, 1].double() @ k["wpk"].double().reshape(row["Cout"], 9, -1)[:, 7, :].t()
            assert chk(y.to(torch.bfloat16)) > 1.0, row
    row, k = grouped
    d = k["stats_delta"].reshape(3, 2, -1)
    assert L.check_stats(k["y"], d, 3) <= 1.0
    bad = d.clone()
    bad[1, :, 5] = d[2, :, 5]                                          # one channel's statistics from the wrong group
    assert L.check_stats(k["y"], bad, 3) > 1.0
