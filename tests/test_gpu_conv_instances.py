"""Every compiled convolution kernel instance, checked per element against float64 (tests/launch_ref.py), with the
instance each call launched taken from torch.profiler and compared with the case table of tests/conv_instances.py.

Outputs the ops wrappers allocate come from a NaN-filled `torch.empty` (conv_instances.NanTorch) and caller-owned
outputs (a wgrad accumulator written with first=True, the conv2d output tensor) are NaN before the call, so an element
a kernel fails to write fails the check. Switches read from the environment once per process run in child processes,
one per group (`python -m tests.test_gpu_conv_instances --group NAME --out FILE`); runtime switches run in-process.
"""
import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile

import pytest
import torch

from tests import conv_instances as CI
from tests import launch_ref as L

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAULT_CASES = ("t9_128_64", "w_256_64_64_ci192", "t9_96_64_mt2")


# ---------------------------------------------------------------------------------------------- one case
def _inputs(c, gen):
    def rnd(*shape, scale=1.0, dtype=torch.bfloat16):
        return (torch.randn(*shape, generator=gen) * scale).to(dtype).cuda()

    from sg2b200 import ops
    o = c.opts
    if c.entry == "conv2d_fprop":
        Ho, Wo = ops.conv2d_out_hw(c.H, c.W, o["kh"], o["kw"], o["stride"], o["ph"], o["pw"])
        return dict(x=rnd(c.B, c.H, c.W, o["x_ctot"]),
                    wpk=rnd(c.Cout, o["kh"] * o["kw"] * c.Cin, scale=(o["kh"] * o["kw"] * c.Cin) ** -0.5),
                    bias=rnd(c.Cout, scale=0.5, dtype=torch.float32),
                    out=torch.full((c.B, Ho, Wo, o["out_ctot"]), math.nan, device="cuda", dtype=torch.bfloat16))
    s1, s2 = ops.pack_shapes(c.kind, c.Cout, c.Cin)
    Ho, Wo = CI.out_hw(c.kind, c.H, c.W)
    d = dict(x=rnd(c.B, c.H, c.W, c.Cin), dy=rnd(c.B, Ho, Wo, c.Cout))
    if c.entry == "conv_fprop":
        d["wpk"] = rnd(*s1, scale=(L.k_fprop(c.kind, c.Cin)) ** -0.5)
        if o.get("bias9"):
            d["bias9"] = rnd(c.B, 9, c.Cout, scale=0.5, dtype=torch.float32)
    elif c.entry == "conv_dgrad":
        d["wpkT"] = rnd(*s2, scale=(L.k_dgrad(c.kind, c.Cout)) ** -0.5)
        if o.get("epi"):
            d["epi"] = (rnd(c.B, c.H, c.W, c.Cin), CI.EPI[o["epi"]])
    else:
        shape = (c.Cout, ops.JOBS[c.kind], c.Cin)
        d["dwpk"] = (torch.full(shape, math.nan, device="cuda") if o.get("first")
                     else torch.randn(shape, generator=gen).cuda())
    return d


def _call(c, d):
    from sg2b200 import ops
    o = c.opts
    if c.entry == "conv_fprop":
        stats = None
        if o.get("stats"):
            stats = torch.zeros(o.get("groups", 1) * 2 * c.Cout, device="cuda", dtype=torch.float64)
        ops.conv_fprop(c.kind, d["x"], d["wpk"], c.Cout, splitk=o.get("splitk"), stats=stats,
                       groups=o.get("groups", 1), act=o.get("act", 0), bias9=d.get("bias9"))
    elif c.entry == "conv_dgrad":
        ops.conv_dgrad(c.kind, d["dy"], d["wpkT"], c.B, c.H, c.W, c.Cin, splitk=o.get("splitk"), epi=d.get("epi"))
    elif c.entry == "conv_wgrad":
        ops.conv_wgrad(c.kind, d["x"], d["dy"], d["dwpk"], splitk=o.get("splitk"), first=bool(o.get("first")))
    else:
        ops.conv2d_fprop(d["x"], c.Cin, d["wpk"], d["bias"], d["out"], c.Cout, o["kh"], o["kw"], o["stride"], o["ph"],
                         o["pw"], o["relu"], o["x_c0"], o["out_c0"])


def _profiled(fn):
    """Run fn under torch.profiler (CUDA activity) -> the conv-family instances it launched (normalised names)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    if not names:
        raise RuntimeError("torch.profiler recorded no CUDA kernels: kernel tracing is unavailable")
    return sorted(CI.conv_family(names))


def run_case(c, keep=False):
    gen = torch.Generator().manual_seed(sum(map(ord, c.name)))
    d = _inputs(c, gen)
    res = dict(instances=[], ratio=None, rows=[], unchecked=[], error=None)
    chk_box = {}

    def body():
        with L.checked(keep=(lambda row: True) if keep else None) as chk:
            chk_box["chk"] = chk
            _call(c, d)

    try:
        res["instances"] = _profiled(body)
    except RuntimeError as e:
        if "kernel tracing" in str(e):
            raise
        res["error"] = str(e)
    torch.cuda.synchronize()
    chk = chk_box.get("chk")
    if chk is not None:
        res["rows"] = chk.rows
        res["unchecked"] = chk.unchecked
        res["ratio"] = max((r["ratio"] for r in chk.rows), default=None)
        if keep:
            res["kept"] = chk.kept
    return res


# ---------------------------------------------------------------------------------------------- one switch group
def run_group(group, keep=()):
    """All cases of one group in this process -> {case name: result}. The process's environment must already match
    the group's environment switches; runtime switches are set here and restored."""
    from sg2b200 import _lib, ops
    spec = CI.GROUPS[group]
    for k, v in spec.get("env", {}).items():
        assert os.environ.get(k) == v, f"group {group} needs {k}={v} in the environment"
    torch.backends.cuda.matmul.allow_tf32 = False
    saved = ops.torch
    ops.torch = CI.NanTorch(torch)
    rt = spec.get("runtime")
    out = {}
    try:
        if rt:
            _lib.call(rt[0], rt[1])
        for c in CI.CASES:
            if c.group == group:
                out[c.name] = run_case(c, keep=c.name in keep)
    finally:
        ops.torch = saved
        if rt:
            _lib.call(rt[0], rt[2])
    return out


_RESULTS = {}


def group_results(group):
    if group not in _RESULTS:
        spec = CI.GROUPS[group]
        if "env" not in spec:
            _RESULTS[group] = run_group(group, keep=FAULT_CASES if group == "default" else ())
        else:
            tmp = tempfile.mkdtemp(prefix="sg2_conv_instances_")
            try:
                path = os.path.join(tmp, f"{group}.json")
                env = dict(os.environ, **spec["env"])
                r = subprocess.run([sys.executable, "-m", "tests.test_gpu_conv_instances", "--group", group, "--out",
                                    path], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
                assert r.returncode == 0, f"group {group}:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
                _RESULTS[group] = json.load(open(path))
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
    return _RESULTS[group]


def _report(group, results):
    lines = []
    for name, r in results.items():
        c = CI.BY_NAME[name]
        ratio = "-" if r["ratio"] is None else f"{r['ratio']:.3f}"
        lines.append(f"{group:>11} {name:<26} {c.entry:<12} {str(CI.KIND_NAMES.get(c.kind, '')):<7} "
                     f"ratio {ratio:>6} {' '.join(r['instances'])}" + (f"  ERROR {r['error']}" if r["error"] else ""))
    return "\n".join(lines)


# ---------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("group", list(CI.GROUPS))
def test_group_cases_within_bound_on_expected_instance(group):
    """Each case of the group: within its float64 bound (ratio <= 1, no NaN), every contraction kernel launched inside
    a checked call, and exactly the expected instance(s) launched. Refused shapes raise the expected error."""
    res = group_results(group)
    print("\n" + _report(group, res))
    bad = []
    for name, r in res.items():
        c = CI.BY_NAME[name]
        if c.refused:
            if not (r["error"] and c.refused in r["error"]):
                bad.append(f"{name}: expected an error containing {c.refused!r}, got {r['error']!r}")
            continue
        if r["error"]:
            bad.append(f"{name}: {r['error']}")
            continue
        if r["unchecked"]:
            bad.append(f"{name}: unchecked launches {r['unchecked']}")
        if not r["rows"] or r["ratio"] is None or not r["ratio"] <= 1.0:
            bad.append(f"{name}: ratio {r['ratio']} over {len(r['rows'])} checked calls")
        if sorted(c.expect) != r["instances"]:
            bad.append(f"{name}: launched {r['instances']}, expected {sorted(c.expect)}")
    assert not bad, "\n".join(bad)


def test_every_compiled_instance_observed_and_checked():
    """The union of the instances launched (and checked) across all groups equals the set of convolution kernels in
    the built library, from cuobjdump -symbols + c++filt."""
    from sg2b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    cxxfilt = shutil.which("c++filt")
    assert os.path.exists(cuobjdump) and cxxfilt, "cuobjdump and c++filt are needed to list the compiled kernels"
    sym = subprocess.run([cuobjdump, "-symbols", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = [ln.split()[-1] for ln in sym.splitlines() if "STO_ENTRY" in ln]
    demangled = subprocess.run([cxxfilt], input="\n".join(mangled), capture_output=True, text=True,
                               check=True).stdout.split("\n")
    compiled = CI.conv_family(demangled)
    assert len(compiled) > 50, sorted(compiled)
    observed, worst = set(), {}
    for g in CI.GROUPS:
        for name, r in group_results(g).items():
            if r["error"] or r["ratio"] is None:
                continue
            for inst in r["instances"]:
                observed.add(inst)
                if inst not in worst or r["ratio"] > worst[inst]["ratio"]:
                    worst[inst] = dict(ratio=r["ratio"], case=name, group=g)
    L.record("instances", {k: worst[k] for k in sorted(worst)}, fname="conv_instance_parity.json")
    L.record("observed", sorted(observed), fname="conv_instance_parity.json")
    L.record("compiled", len(compiled), fname="conv_instance_parity.json")
    print(f"\n{len(observed & compiled)} of {len(compiled)} compiled convolution instances observed and checked")
    assert compiled - observed == set(), f"never launched: {sorted(compiled - observed)}"
    assert observed - compiled == set(), f"launched but not in the library: {sorted(observed - compiled)}"


def _fault(v):
    v = v.float()
    return v + 0.25 + 0.5 * v.abs()             # off by at least 0.25 and by half of its value


def test_checker_rejects_faults_at_the_new_edges():
    """Seeded faults in real kernel outputs (host-side copies): one element of the last partial pixel tile of a 24 x 20
    map, one column just past a 64-wide boundary of a Cin = 192 gather wgrad, one element of the upper 96-wide half
    of an N = 192 ring-mode (mt = 2) output."""
    res = group_results("default")

    def kept(name):
        r = res[name]
        assert r["error"] is None and r.get("kept"), name
        return r["kept"][0]

    row, k = kept("t9_128_64")
    kind = getattr(L, row["kind"])

    def chk_f(y, row=row, k=k, kind=kind):
        return L.check_fprop(kind, k["x"], k["wpk"], y, row["Cout"], k["splits"], k["act"], k["bias9"])

    assert chk_f(k["y"]) <= 1.0
    y = k["y"].clone()
    y[-1, 23, 19, 5] = _fault(y[-1, 23, 19, 5])                      # last row / column of the last partial tile
    assert chk_f(y) > 1.0

    row, k = kept("w_256_64_64_ci192")
    kind = getattr(L, row["kind"])
    assert row["Cin"] == 192
    assert L.check_wgrad(kind, k["x"], k["dy"], k["dwpk"], k["old"], k["slabs"]) <= 1.0
    dw = k["dwpk"].clone()
    dw[3, 4, 64] = _fault(dw[3, 4, 64])                              # first column of the second 64-wide chunk
    assert L.check_wgrad(kind, k["x"], k["dy"], dw, k["old"], k["slabs"]) > 1.0

    row, k = kept("t9_96_64_mt2")
    kind = getattr(L, row["kind"])
    assert row["Cout"] == 192
    assert chk_f(k["y"], row, k, kind) <= 1.0
    y = k["y"].clone()
    y[7, 40, 33, 96 + 17] = _fault(y[7, 40, 33, 96 + 17])
    assert chk_f(y, row, k, kind) > 1.0


def _jsonable(results):
    out = {}
    for name, r in results.items():
        r = {k: v for k, v in r.items() if k != "kept"}
        r["rows"] = [{k: v for k, v in row.items()} for row in r["rows"]]
        out[name] = r
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--group", required=True, choices=list(CI.GROUPS))
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    res = run_group(a.group)
    json.dump(_jsonable(res), open(a.out, "w"), default=str)
    print(_report(a.group, res))
