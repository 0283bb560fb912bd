"""The case table of tests/conv_instances.py against the kernels csrc/conv.cu compiles, without a GPU: every compiled
instance is claimed by some case, every expected instance exists, every (family, entry, kind) combination the
dispatcher produces is exercised, each case's shape meets the entry's documented preconditions unless it is marked as
refused, and the NaN-poisoning stand-in for torch behaves."""
import math
import os
import shutil
import subprocess

import pytest
import torch

from tests import conv_instances as CI

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def compiled(tmp_path_factory):
    """Kernel instances of csrc/conv.cu cross-compiled for sm_100a with the library's flags (about a minute)."""
    import sg2b200.build as build
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    cxxfilt = shutil.which("c++filt")
    if not (os.path.exists(nvcc) and os.path.exists(cuobjdump) and cxxfilt):
        pytest.skip("needs nvcc, cuobjdump and c++filt")
    obj = str(tmp_path_factory.mktemp("conv") / "conv.o")
    r = subprocess.run([nvcc, *build.NVCC_FLAGS, "-c", os.path.join(build.CSRC, "conv.cu"), "-o", obj],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    sym = subprocess.run([cuobjdump, "-symbols", obj], capture_output=True, text=True, check=True).stdout
    mangled = [ln.split()[-1] for ln in sym.splitlines() if "STO_ENTRY" in ln]
    names = subprocess.run([cxxfilt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    return CI.conv_family(names.split("\n"))


def test_every_compiled_instance_claimed_and_every_expected_instance_compiled(compiled):
    claimed = {i for c in CI.CASES for i in c.expect}
    assert len(compiled) > 50, sorted(compiled)
    assert compiled - claimed == set(), f"compiled but claimed by no case: {sorted(compiled - claimed)}"
    assert claimed - compiled == set(), f"expected by a case but not compiled: {sorted(claimed - compiled)}"


def test_every_dispatch_combination_exercised():
    missing = CI.REQUIRED_COMBOS - CI.combos()
    assert not missing, sorted(missing, key=str)


def test_groups_and_instance_names_well_formed():
    assert {c.group for c in CI.CASES} == set(CI.GROUPS)
    for c in CI.CASES:
        assert bool(c.refused) != bool(c.expect), c.name      # a case either launches named instances or is refused
        for inst in c.expect:
            assert CI.CONV_FAMILY.match(inst) and CI.normalise(inst) == inst, (c.name, inst)
            CI.family(inst)
        if c.entry != "conv2d_fprop":
            assert c.kind in CI.KIND_NAMES, c.name
    for spec in CI.GROUPS.values():
        assert set(spec) <= {"env", "runtime"}


def test_cases_meet_preconditions_unless_refused():
    for c in CI.CASES:
        v = CI.violations(c)
        if c.refused:
            assert v, f"{c.name} is marked refused but meets every documented precondition"
        else:
            assert not v, f"{c.name}: {v}"


def test_precondition_validator_rejects_each_violation():
    base = CI.BY_NAME["t9_64_64"]
    assert CI.violations(base) == []
    bad = [base._replace(Cin=24), base._replace(kind=CI.CONV4S2, H=25),
           base._replace(H=6, W=6),                                     # gather grid, no 128-pixel box
           base._replace(opts=dict(base.opts, act=CI.ACT_LRELU)),      # activation with statistics
           base._replace(H=4, W=4),                                     # region bias on a gather grid
           base._replace(B=3, opts=dict(base.opts, groups=2))]
    for c in bad:
        assert CI.violations(c), c
    w = CI.BY_NAME["w_64_32_64"]
    assert CI.violations(w) == [] and CI.violations(w._replace(Cin=80)) and CI.violations(w._replace(Cout=48))
    c2 = CI.BY_NAME["c2_1x7"]
    assert CI.violations(c2) == []
    for opts in (dict(kh=7, kw=7), dict(stride=3), dict(ph=1), dict(out_c0=200), dict(x_c0=4, x_ctot=68)):
        assert CI.violations(c2._replace(opts=dict(c2.opts, **opts))), opts


def test_pick_tile_matches_the_dispatcher():
    assert CI.pick_tile(4, 4, 128) == (4, 4, 8)
    assert CI.pick_tile(24, 12, 128) == (16, 8, 1)
    assert CI.pick_tile(300, 1, 128) == (128, 1, 1)
    assert CI.pick_tile(1, 1, 128) == (1, 1, 128)
    assert CI.pick_tile(6, 6, 128) is None
    assert CI.pick_tile(300, 1, 64) == (64, 1, 1)


def test_kernel_name_normalisation():
    assert CI.normalise("void sg2::tile_conv_kernel<128, 16, 4>(sg2::TileParams)") == CI.T(128, 16, 4)
    assert CI.normalise("void sg2::igemm_fprop_pair_kernel<256, 64, true>(sg2::FpropParams)") == CI.P(True)
    assert CI.normalise("sg2::igemm_wgrad_pair_kernel(sg2::WgradParams)") == CI.WP
    assert CI.conv_family(["void sg2::bn_stats_kernel(int)", "void sg2::tile_wgrad_kernel(sg2::TileWgradParams)",
                           "at::native::vectorized_elementwise_kernel<4>(int)"]) == {CI.TW}


def test_nan_torch_poisons_float_allocations_only():
    t = CI.NanTorch(torch)
    for dt in (torch.float32, torch.bfloat16, torch.float64):
        a = t.empty((3, 5), dtype=dt)
        assert a.dtype == dt and a.shape == (3, 5) and bool(torch.isnan(a).all())
        b = t.empty_like(torch.zeros(4, dtype=dt))
        assert bool(torch.isnan(b).all())
    assert t.empty(7, dtype=torch.int32).dtype == torch.int32          # integers are left alone
    assert t.float32 is torch.float32 and t.zeros(3).sum() == 0        # everything else is torch
    assert bool(torch.isnan(t.empty(2, 2)).all()) and math.isnan(float(t.empty(1)))
