"""Case table over the dispatch space of the convolution library (csrc/conv.cu): which compiled kernel instance each
public entry point selects for which shape, split factor, epilogue and switch.

Every case names the entry (conv_fprop, conv_dgrad, conv_wgrad, conv2d_fprop), the kind, B, H, W, Cin, Cout, its
options, the switch group it runs in and the instance(s) it is expected to launch. tests/test_gpu_conv_instances.py runs
each case inside tests/launch_ref.py's per-element float64 checker, records the instances it launched with
torch.profiler and compares them with this table; tests/test_conv_instances_host.py checks, without a GPU, that every
instance compiled from csrc/conv.cu is claimed by some case and that every case's shape meets the entry's documented
preconditions (or is marked as refused).

Instance names are the demangled kernel names without `void ` and without the argument list, as c++filt prints the
symbols cuobjdump lists and as torch.profiler reports the launched kernels.
"""
import math
import re
from collections import namedtuple

CONV3, UPCONV, CONV4S2, GEMM = 0, 1, 2, 3
KIND_NAMES = {CONV3: "CONV3", UPCONV: "UPCONV", CONV4S2: "CONV4S2", GEMM: "GEMM"}
EPI = {"add": 1, "mask": 2}
ACT_LRELU = 2

# kernels of the convolution library (the other kernels of libsg2b200.so are elementwise / BatchNorm / linears)
CONV_FAMILY = re.compile(r"^sg2::(tile_conv_kernel|tile_wgrad_kernel|igemm_fprop_kernel|igemm_fprop_cluster_kernel|"
                         r"igemm_fprop_pair_kernel|igemm_wgrad_kernel|igemm_wgrad_pair_kernel)\b")


def normalise(name):
    """'void sg2::f<1, 2>(sg2::P)' -> 'sg2::f<1, 2>'."""
    name = name.strip()
    if name.startswith("void "):
        name = name[5:]
    depth = 0
    for i, ch in enumerate(name):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            return name[:i].strip()
    return name


def conv_family(names):
    return {n for n in (normalise(x) for x in names) if CONV_FAMILY.match(n)}


# ---------------------------------------------------------------------------------------------- instance names
def T(bn, bk, nt):
    return f"sg2::tile_conv_kernel<{bn}, {bk}, {nt}>"


def G(bn, bk, mt=1):
    return f"sg2::igemm_fprop_kernel<{bn}, {bk}, {mt}>"


def CL(bn, bk, mt=1):
    return f"sg2::igemm_fprop_cluster_kernel<{bn}, {bk}, {mt}>"


def P(direct):
    return f"sg2::igemm_fprop_pair_kernel<256, 64, {'true' if direct else 'false'}>"


def WG(bn, cwa, cwb):
    return f"sg2::igemm_wgrad_kernel<{bn}, {cwa}, {cwb}>"


WP = "sg2::igemm_wgrad_pair_kernel"
TW = "sg2::tile_wgrad_kernel"


def family(instance):
    return {"tile_conv_kernel": "tile", "igemm_fprop_kernel": "gather", "igemm_fprop_cluster_kernel": "cluster",
            "igemm_fprop_pair_kernel": "pair", "igemm_wgrad_kernel": "wgrad_gather", "tile_wgrad_kernel": "wgrad_tile",
            "igemm_wgrad_pair_kernel": "wgrad_pair"}[re.match(r"sg2::(\w+)", instance).group(1)]


# ---------------------------------------------------------------------------------------------- switch groups
# runtime switches run in the test process (and are restored); environment switches are read once per process, so
# each of those groups runs in a child process of its own
GROUPS = {
    "default": {},
    "pair_off": {"runtime": ("sg2_set_pair_kernels", 0, -1)},
    "sm_reserve": {"runtime": ("sg2_set_sm_reserve", 8, 0)},
    "mt2": {"env": {"SG2_IGEMM_MT2": "1", "SG2_PAIR": "0"}},
    "cluster4": {"env": {"SG2_CLUSTER_SPLITK": "4"}},
    "atomic": {"env": {"SG2_DETERMINISTIC": "0"}},
    "gather_only": {"env": {"SG2_TILE": "0", "SG2_TILE_WGRAD": "0"}},
    "knobs": {"env": {"SG2_WGRAD_MERGE": "0", "SG2_RES_HALF": "1", "SG2_PAIR_WGRAD": "0"}},
}

Case = namedtuple("Case", "name entry kind B H W Cin Cout opts group expect refused")
CASES = []


def _add(name, entry, kind, B, H, W, Cin, Cout, expect=(), group="default", refused=None, **opts):
    if entry in ("fprop", "dgrad"):
        opts.setdefault("splitk", 1)
    CASES.append(Case(name, "conv_" + entry if entry != "conv2d" else "conv2d_fprop", kind, B, H, W, Cin, Cout, opts,
                      group, (expect,) if isinstance(expect, str) else tuple(expect), refused))


F = lambda name, *a, **k: _add(name, "fprop", *a, **k)       # noqa: E731
D = lambda name, *a, **k: _add(name, "dgrad", *a, **k)       # noqa: E731
W_ = lambda name, *a, **k: _add(name, "wgrad", *a, **k)      # noqa: E731


def C2(name, B, H, W, Cin, Cout, expect, kh=3, kw=3, stride=1, ph=1, pw=1, relu=True, x_c0=0, out_c0=0, x_ctot=None,
       out_ctot=None, refused=None):
    _add(name, "conv2d", None, B, H, W, Cin, Cout, expect, refused=refused, kh=kh, kw=kw, stride=stride, ph=ph, pw=pw,
         relu=relu, x_c0=x_c0, out_c0=out_c0, x_ctot=x_ctot or x_c0 + Cin, out_ctot=out_ctot or out_c0 + Cout)


# ---- tile-resident kernel, 9 taps (CONV3 fprop / dgrad). 24 x 20 maps: partial 16 x 8 tiles in both directions.
# dgrad: N = Cin (the tile width), K = Cout (BK).
F("t9_256_16", CONV3, 1, 24, 20, 16, 256, T(256, 16, 9))
F("t9_256_32", CONV3, 1, 24, 20, 32, 256, T(256, 32, 9))
F("t9_256_64_ring", CONV3, 1, 24, 20, 64, 256, T(256, 64, 9))                 # 288 KB of weights: ring, one tile
D("t9_128_16", CONV3, 1, 24, 20, 128, 16, T(128, 16, 9))
F("t9_128_32", CONV3, 1, 24, 20, 32, 128, T(128, 32, 9), stats=True)
F("t9_128_64", CONV3, 2, 24, 20, 64, 128, T(128, 64, 9))
F("t9_64_16", CONV3, 1, 24, 20, 16, 64, T(64, 16, 9), act=ACT_LRELU)
D("t9_64_32", CONV3, 1, 24, 20, 64, 32, T(64, 32, 9), epi="add")
F("t9_64_64", CONV3, 2, 24, 20, 64, 64, T(64, 64, 9), bias9=True, stats=True)
F("t9_32_16", CONV3, 1, 24, 20, 16, 32, T(32, 16, 9))
D("t9_32_32", CONV3, 1, 24, 20, 32, 32, T(32, 32, 9), epi="mask")
F("t9_32_64", CONV3, 1, 24, 20, 64, 32, T(32, 64, 9))
F("t9_16_16", CONV3, 1, 24, 20, 16, 16, T(16, 16, 9))
D("t9_16_32", CONV3, 1, 24, 20, 16, 32, T(16, 32, 9))
F("t9_16_64", CONV3, 1, 24, 20, 64, 16, T(16, 64, 9))
F("t9_160_32_resident", CONV3, 1, 24, 20, 32, 160, T(160, 32, 9))
F("t9_192_32_resident", CONV3, 3, 24, 20, 32, 192, T(192, 32, 9), stats=True, groups=3)
F("t9_160_64_ring", CONV3, 1, 24, 20, 64, 160, T(160, 64, 9))
D("t9_192_64_ring", CONV3, 1, 24, 20, 192, 64, T(192, 64, 9))
# ring mode with two pixel tiles per unit (mt = 2): >= 2 x 74 units of 2 tiles (10 x 32 tiles of a 64 x 64 map)
F("t9_96_64_mt2", CONV3, 10, 64, 64, 64, 192, T(96, 64, 9))
F("t9_80_64_mt2", CONV3, 10, 64, 64, 64, 160, T(80, 64, 9))
F("t9_96_32_mt2", CONV3, 10, 64, 64, 96, 192, T(96, 32, 9))
D("t9_80_32_mt2", CONV3, 10, 64, 64, 160, 96, T(80, 32, 9))
F("t9_128_64_mt2", CONV3, 10, 64, 64, 64, 256, T(128, 64, 9))

# ---- tile-resident kernel, 4 taps per source: UPCONV fprop (4 parity groups), CONV4S2 fprop (4 parity sources),
# UPCONV dgrad (4 sources), CONV4S2 dgrad (4 groups). Output grids of 24 x 20.
F("t4_256_64", UPCONV, 1, 24, 20, 64, 256, T(256, 64, 4))
F("t4_256_16", UPCONV, 1, 24, 20, 16, 256, T(256, 16, 4))
D("t4_256_32", CONV4S2, 1, 48, 40, 256, 32, T(256, 32, 4))
F("t4_128_64_ring", CONV4S2, 1, 48, 40, 64, 128, T(128, 64, 4))
D("t4_128_32", UPCONV, 1, 24, 20, 128, 32, T(128, 32, 4))
D("t4_128_16", UPCONV, 1, 24, 20, 128, 16, T(128, 16, 4), epi="add")
D("t4_64_64", CONV4S2, 1, 48, 40, 64, 64, T(64, 64, 4), epi="mask")
F("t4_64_32", CONV4S2, 1, 48, 40, 32, 64, T(64, 32, 4), stats=True)
F("t4_64_16", UPCONV, 1, 24, 20, 16, 64, T(64, 16, 4))
D("t4_32_64", UPCONV, 1, 24, 20, 32, 64, T(32, 64, 4))
F("t4_32_32", UPCONV, 1, 24, 20, 32, 32, T(32, 32, 4))
F("t4_32_16", CONV4S2, 1, 48, 40, 16, 32, T(32, 16, 4))
D("t4_16_64", CONV4S2, 1, 48, 40, 16, 64, T(16, 64, 4))
D("t4_16_32", UPCONV, 1, 24, 20, 16, 32, T(16, 32, 4))
F("t4_16_16", UPCONV, 1, 24, 20, 16, 16, T(16, 16, 4))
F("t4_160_64", UPCONV, 1, 24, 20, 64, 160, T(160, 64, 4))
D("t4_160_32", CONV4S2, 1, 48, 40, 160, 32, T(160, 32, 4))
F("t4_192_64", UPCONV, 1, 24, 20, 64, 192, T(192, 64, 4))
D("t4_192_32", CONV4S2, 1, 48, 40, 192, 32, T(192, 32, 4))
F("t4_96_64_mt2", UPCONV, 9, 32, 32, 128, 192, T(96, 64, 4))
F("t4_96_32_mt2", UPCONV, 9, 32, 32, 160, 192, T(96, 32, 4))
F("t4_80_64_mt2", UPCONV, 9, 32, 32, 128, 160, T(80, 64, 4))
F("t4_80_32_mt2", UPCONV, 9, 32, 32, 160, 160, T(80, 32, 4))
# ---- tile-resident 1-tap GEMM tiles (64 -> 64)
F("t1_gemm", GEMM, 1, 16, 8, 64, 64, T(64, 64, 1))
D("t1_gemm_dgrad", GEMM, 2, 24, 20, 64, 64, T(64, 64, 1))

# ---- plain gather kernel through conv_fprop / conv_dgrad: grids below 16 x 8, partial 128-row boxes
F("g_conv3_b3", CONV3, 3, 4, 4, 64, 64, G(64, 64))                           # 48 of 128 rows
F("g_conv3_12x24", CONV3, 1, 12, 24, 64, 128, G(128, 64))                    # 16 x 8 boxes, partial in x and y
F("g_conv3_1x1", CONV3, 3, 1, 1, 32, 32, G(32, 32))
F("g_b1_1x1", CONV3, 1, 1, 1, 16, 16, G(16, 16))
D("g_conv3_dgrad", CONV3, 3, 4, 4, 128, 64, G(128, 64))
F("g_up", UPCONV, 2, 4, 4, 64, 64, G(64, 64))
D("g_up_dgrad", UPCONV, 2, 4, 4, 64, 32, G(64, 32))
F("g_s2", CONV4S2, 2, 8, 8, 32, 64, G(64, 32))
D("g_s2_dgrad", CONV4S2, 2, 8, 8, 64, 64, G(64, 64))
F("g_gemm", GEMM, 1, 1, 300, 64, 64, G(64, 64))                              # last box 44 rows
D("g_gemm_dgrad", GEMM, 1, 1, 300, 32, 64, G(32, 64))
F("g_stats_groups_fused", CONV3, 24, 4, 4, 64, 64, G(64, 64), stats=True, groups=3)
F("g_stats_straddle", CONV3, 6, 4, 4, 64, 64, G(64, 64), stats=True, groups=3)   # 8-image box over 2-image groups
D("g_epi_nofuse", CONV3, 3, 4, 4, 64, 64, G(64, 64), epi="add")                 # gather: separate epilogue kernel

# ---- CTA pairs (256-wide tiles over two SMs); an odd tile count runs a phantom peer
F("p_direct_odd", CONV3, 24, 4, 4, 64, 256, P(True), stats=True, groups=3)
D("p_direct_dgrad", CONV3, 20, 4, 4, 256, 64, P(True), epi="mask")
D("p_direct_up_dgrad", UPCONV, 24, 4, 4, 256, 64, P(True))
D("p_direct_s2_dgrad", CONV4S2, 24, 8, 8, 256, 64, P(True))
F("p_direct_gemm", GEMM, 1, 1, 512, 64, 256, P(True))
D("p_direct_gemm_dgrad", GEMM, 1, 1, 512, 256, 64, P(True))
F("p_split_s2", CONV4S2, 12, 16, 16, 128, 256, P(False), splitk=2)
F("p_split_up", UPCONV, 24, 4, 4, 256, 256, P(False), splitk=2)

# ---- split-K inside a thread-block cluster (1 < split <= SG2_CLUSTER_SPLITK)
F("c_128_stats", CONV3, 2, 4, 4, 64, 128, CL(128, 64), splitk=2, stats=True)
F("c_64_up", UPCONV, 2, 4, 4, 64, 64, CL(64, 64), splitk=2)
D("c_64_up_dgrad", UPCONV, 2, 4, 4, 64, 64, CL(64, 64), splitk=2)
D("c_256_s2_dgrad", CONV4S2, 2, 8, 8, 256, 64, CL(256, 64), splitk=2)            # one gather tile: no pair
F("c_256_single_tile", CONV3, 1, 4, 4, 64, 256, CL(256, 64), splitk=2)
D("c_epi_add", CONV3, 2, 4, 4, 128, 64, CL(128, 64), splitk=2, epi="add")
F("c_gemm", GEMM, 1, 1, 256, 128, 64, CL(64, 64), splitk=2)
D("c_gemm_dgrad", GEMM, 1, 1, 256, 64, 128, CL(64, 64), splitk=2)
F("c_s2", CONV4S2, 2, 8, 8, 64, 128, CL(128, 64), splitk=2)
F("c_auto", CONV3, 2, 4, 4, 512, 64, CL(64, 64), splitk=None)                   # _auto_split picks 2
# NoFuse retries onto the slab path: statistics groups straddled by the 8-image box, no 192-wide cluster instance
F("c_straddle_to_slabs", CONV3, 6, 4, 4, 64, 64, G(64, 64), splitk=2, stats=True, groups=3)
F("c_192_to_slabs", CONV3, 2, 4, 4, 64, 192, G(192, 64), splitk=2)

# ---- split-K slabs (fp32 per split) + the ordered splitk_finish pass
F("s_stats", CONV3, 2, 8, 8, 64, 64, G(64, 64), splitk=3, stats=True)
F("s_stats_groups", CONV3, 6, 4, 4, 64, 64, G(64, 64), splitk=3, stats=True, groups=3)
D("s_epi_add", CONV3, 2, 8, 8, 64, 64, G(64, 64), splitk=3, epi="add")
D("s_epi_mask", UPCONV, 2, 4, 4, 64, 128, G(64, 64), splitk=4, epi="mask")
F("s_clamped", CONV3, 2, 4, 4, 16, 32, G(32, 16), splitk=50)                     # 9 K blocks: split 9
F("s_up", UPCONV, 2, 4, 4, 128, 128, G(128, 64), splitk=3)

# ---- gather weight gradient: every (BN, CWA, CWB); Cin not a multiple of BN, Cout < 128 and 128 < Cout < 256
W_("w_16_32_16", CONV3, 2, 4, 4, 16, 32, WG(16, 32, 16), first=True)
W_("w_16_64_16", CONV3, 2, 4, 4, 16, 64, WG(16, 64, 16))
W_("w_32_32_32", CONV3, 2, 4, 4, 32, 32, WG(32, 32, 32), first=True)
W_("w_32_64_32", CONV3, 2, 4, 4, 32, 64, WG(32, 64, 32))
W_("w_64_32_64", CONV3, 2, 4, 4, 64, 32, WG(64, 32, 64), first=True)
W_("w_64_64_64_up", UPCONV, 2, 4, 4, 64, 64, WG(64, 64, 64))
W_("w_128_32_32", CONV3, 2, 4, 4, 96, 32, WG(128, 32, 32), first=True)
W_("w_128_64_32_s2", CONV4S2, 2, 8, 8, 96, 64, WG(128, 64, 32))
W_("w_128_32_64_co96", CONV3, 2, 4, 4, 128, 96, WG(128, 32, 64), first=True)
W_("w_128_64_64_co192", CONV3, 2, 4, 4, 128, 192, WG(128, 64, 64))
W_("w_256_64_32_ci160", CONV3, 2, 4, 4, 160, 64, WG(256, 64, 32), first=True)
W_("w_256_32_32_ci160", CONV3, 2, 4, 4, 160, 96, WG(256, 32, 32))
W_("w_256_32_64_ci320", CONV3, 2, 4, 4, 320, 32, WG(256, 32, 64), first=True)
W_("w_256_64_64_ci192", CONV3, 2, 4, 4, 192, 64, WG(256, 64, 64), first=True)
W_("w_256_32_64_s2_ci192", CONV4S2, 2, 8, 8, 192, 96, WG(256, 32, 64))
W_("w_gemm", GEMM, 1, 1, 300, 64, 64, WG(64, 64, 64), first=True)
W_("w_slabs_first", CONV3, 2, 8, 8, 64, 64, WG(64, 64, 64), splitk=4, first=True)
W_("w_pair", CONV3, 2, 4, 4, 256, 256, WP, first=True)
W_("w_pair_up", UPCONV, 2, 4, 4, 256, 256, WP)
W_("w_pair_s2", CONV4S2, 2, 8, 8, 256, 256, WP)
W_("w_pair_gemm", GEMM, 1, 1, 256, 256, 256, WP)
# ---- tile-resident weight gradient: merge3 on (BN 64) and off (BN 128), CTA lanes > 1, parity sources
W_("tw_merge3", CONV3, 2, 32, 16, 64, 64, TW, first=True)
W_("tw_no_merge", CONV3, 2, 32, 16, 128, 64, TW)
W_("tw_up", UPCONV, 1, 24, 20, 32, 64, TW, first=True)
W_("tw_s2", CONV4S2, 1, 48, 40, 64, 32, TW)
W_("tw_gemm", GEMM, 1, 16, 8, 64, 64, TW, first=True)
W_("tw_co96", CONV3, 2, 24, 20, 64, 96, TW)
W_("tw_to_gather_co192", CONV3, 2, 16, 16, 64, 192, WG(64, 64, 64))          # Cout > 128 on few pixels: gather

# ---- general convolution (Inception): every conv2d_bn choice, flat 1x1, stride 2, 1x7 / 7x1 / 5x5 / 32 taps, slices
C2("c2_1x1_p35", 1, 5, 7, 64, 16, G(16, 64), kh=1, kw=1, ph=0, pw=0)
C2("c2_1x1_p297_slices", 3, 9, 11, 32, 24, G(32, 32), kh=1, kw=1, ph=0, pw=0, x_c0=16, x_ctot=56, out_c0=8,
   out_ctot=40)
C2("c2_s2_odd", 2, 17, 15, 16, 48, G(64, 16), stride=2, ph=0, pw=0)
C2("c2_s2_pad_odd", 2, 13, 11, 32, 64, G(64, 32), stride=2)
C2("c2_1x7", 2, 9, 9, 64, 128, G(128, 64), kh=1, kw=7, ph=0, pw=3, out_c0=64, out_ctot=256)
C2("c2_7x1", 2, 9, 9, 32, 120, G(128, 32), kh=7, kw=1, ph=3, pw=0, x_c0=32, x_ctot=96)
C2("c2_5x5", 2, 10, 10, 16, 96, G(128, 16), kh=5, kw=5, ph=2, pw=2)
C2("c2_32taps", 2, 8, 12, 16, 32, G(32, 16), kh=4, kw=8, ph=1, pw=3)
C2("c2_160_64", 2, 9, 9, 64, 160, G(160, 64))
C2("c2_144_on_160_32", 2, 9, 9, 32, 144, G(160, 32))
C2("c2_176_on_192_64", 2, 9, 9, 64, 176, G(192, 64))
C2("c2_192_32", 2, 9, 9, 32, 192, G(192, 32), relu=False)
C2("c2_256_64", 2, 9, 9, 64, 256, G(256, 64), ph=0, pw=0)
C2("c2_224_on_256_32", 2, 9, 9, 32, 224, G(256, 32))
C2("c2_200_on_256_16", 2, 9, 9, 16, 200, G(256, 16))
C2("c2_320_on_160_64", 2, 9, 9, 64, 320, G(160, 64))                          # above 256: two 160-wide tiles
C2("c2_384_on_192_32", 2, 9, 9, 32, 384, G(192, 32))
C2("c2_288_on_128_16", 2, 9, 9, 16, 288, G(128, 16))
C2("c2_64_64_slices", 2, 9, 9, 64, 64, G(64, 64), x_c0=64, x_ctot=192, out_c0=32, out_ctot=128)
C2("c2_32_64", 2, 9, 9, 64, 32, G(32, 64))
C2("c2_16_32", 2, 9, 9, 32, 16, G(16, 32))
C2("c2_8_on_16_16", 2, 6, 6, 16, 8, G(16, 16), relu=False)
C2("c2_3x3_on_1x1", 3, 1, 1, 32, 64, G(64, 32))

# ---- shapes the entry points refuse (an error, never a silent result)
W_("r_wgrad_cin48", CONV3, 2, 4, 4, 48, 64, refused="no wgrad instance")        # no CWB = 16 instance for BN >= 64
F("r_bias9_gather", CONV3, 2, 4, 4, 64, 64, refused="region bias", bias9=True)
F("r_cin24", CONV3, 2, 4, 4, 24, 64, refused="multiple of 16")
D("r_dgrad_cout24", CONV3, 2, 4, 4, 64, 24, refused="multiple of 16")
C2("r_conv2d_cin24", 2, 9, 9, 24, 64, (), refused="multiple of 16")
F("r_160_bk16", CONV3, 2, 4, 4, 48, 160, refused="no fprop instance")           # BK = 16 has no 160-wide tile
F("r_map6x6", CONV3, 2, 6, 6, 64, 64, refused="no 128-pixel tile")             # 36-pixel images do not tile 128 rows

# ---- runtime switches (in-process)
F("po_plain_256", CONV3, 24, 4, 4, 64, 256, G(256, 64), group="pair_off")
F("po_cluster_256", CONV3, 24, 4, 4, 64, 256, CL(256, 64), group="pair_off", splitk=2)
D("po_dgrad_256", CONV3, 20, 4, 4, 256, 64, G(256, 64), group="pair_off")
W_("po_wgrad_256", CONV3, 2, 4, 4, 256, 256, WG(256, 64, 64), group="pair_off", first=True)
F("sr_mt2", CONV3, 10, 64, 64, 64, 192, T(96, 64, 9), group="sm_reserve")
W_("sr_tile_wgrad", CONV3, 2, 32, 16, 64, 64, TW, group="sm_reserve", first=True)
F("sr_pair", CONV3, 24, 4, 4, 64, 256, P(True), group="sm_reserve")

# ---- environment switches (one child process per group)
F("m_plain_mt2", CONV3, 24, 4, 4, 64, 256, G(256, 64, 2), group="mt2")
F("m_cluster_mt2", CONV3, 24, 4, 4, 64, 256, CL(256, 64, 2), group="mt2", splitk=2, stats=True)
D("m_slabs_mt2", CONV3, 20, 4, 4, 256, 64, G(256, 64, 2), group="mt2", splitk=3, epi="add")
F("k4_split3", CONV3, 2, 4, 4, 64, 128, CL(128, 64), group="cluster4", splitk=3, stats=True)
F("k4_split4_s2", CONV4S2, 2, 8, 8, 64, 64, CL(64, 64), group="cluster4", splitk=4)
D("k4_split4_dgrad", CONV3, 2, 4, 4, 256, 64, CL(256, 64), group="cluster4", splitk=4, epi="mask")
F("k4_pair_split4", UPCONV, 24, 4, 4, 256, 256, P(False), group="cluster4", splitk=4)
F("a_split3_stats", CONV3, 2, 4, 4, 64, 64, G(64, 64), group="atomic", splitk=3, stats=True)
F("a_split2", CONV3, 2, 4, 4, 64, 128, G(128, 64), group="atomic", splitk=2)
D("a_dgrad_epi", CONV3, 2, 8, 8, 64, 64, G(64, 64), group="atomic", splitk=3, epi="add")
W_("a_wgrad_gather", CONV3, 2, 8, 8, 64, 64, WG(64, 64, 64), group="atomic", splitk=2)
W_("a_wgrad_tile", CONV3, 2, 32, 16, 64, 64, TW, group="atomic")
W_("a_wgrad_pair", CONV3, 2, 4, 4, 256, 256, WP, group="atomic")
F("go_conv3", CONV3, 1, 24, 20, 64, 64, G(64, 64), group="gather_only")
F("go_up", UPCONV, 1, 24, 20, 64, 64, G(64, 64), group="gather_only")
D("go_s2_dgrad", CONV4S2, 1, 48, 40, 64, 64, G(64, 64), group="gather_only")
W_("go_wgrad", CONV3, 1, 24, 20, 64, 64, WG(64, 64, 64), group="gather_only", first=True)
W_("go_wgrad_ci160", CONV3, 1, 24, 20, 160, 64, WG(256, 64, 32), group="gather_only")
W_("kn_merge_off", CONV3, 2, 32, 16, 64, 64, TW, group="knobs", first=True)
F("kn_res_half", CONV4S2, 1, 48, 40, 64, 128, T(64, 64, 4), group="knobs")
W_("kn_pair_wgrad_off", CONV3, 2, 4, 4, 256, 256, WG(256, 64, 64), group="knobs")

BY_NAME = {c.name: c for c in CASES}
assert len(BY_NAME) == len(CASES), "case names must be unique"

# (family, entry, kind) combinations the dispatcher can produce; each must be exercised by some case
REQUIRED_COMBOS = (
    {("tile", e, k) for e in ("conv_fprop", "conv_dgrad") for k in (CONV3, UPCONV, CONV4S2, GEMM)}
    | {("gather", e, k) for e in ("conv_fprop", "conv_dgrad") for k in (CONV3, UPCONV, CONV4S2, GEMM)}
    | {("gather", "conv2d_fprop", None)}
    | {("cluster", e, k) for e in ("conv_fprop", "conv_dgrad") for k in (CONV3, UPCONV, CONV4S2, GEMM)}
    | {("pair", e, k) for e in ("conv_fprop", "conv_dgrad") for k in (CONV3, UPCONV, CONV4S2, GEMM)}
    | {(f, "conv_wgrad", k) for f in ("wgrad_gather", "wgrad_tile", "wgrad_pair") for k in (CONV3, UPCONV, CONV4S2, GEMM)}
)


def combos(cases=None):
    out = set()
    for c in cases or CASES:
        for inst in c.expect:
            out.add((family(inst), c.entry, c.kind))
    return out


# ---------------------------------------------------------------------------------------------- preconditions
def out_hw(kind, H, W):
    if kind == UPCONV:
        return 2 * H, 2 * W
    if kind == CONV4S2:
        return H // 2, W // 2
    return H, W


def pick_tile(Wg, Hg, npix):
    """conv.cu pick_tile: the (tw, th, nb) box of exactly npix pixels over a Wg x Hg grid, or None."""
    w = min(Wg, npix) if Hg == 1 else min(Wg, 16)
    h = min(npix // w, Hg) if w > 0 else 0
    if w <= 0 or h <= 0 or npix % (w * h):
        return None
    return w, h, npix // (w * h)


def _grid(c):
    """Per-group output grid of a conv_fprop / conv_dgrad / conv_wgrad launch (conv.cu Wg x Hg)."""
    if c.kind == CONV4S2:
        return c.W // 2, c.H // 2
    return c.W, c.H


def violations(c):
    """Documented preconditions (include/sg2b200.h, conv.cu) this case breaks; empty for a valid shape."""
    o, bad = c.opts, []
    if min(c.B, c.H, c.W) < 1:
        bad.append("empty input")
    if c.entry == "conv2d_fprop":
        kh, kw, s, ph, pw = o["kh"], o["kw"], o["stride"], o["ph"], o["pw"]
        if c.Cin < 16 or c.Cin % 16:
            bad.append("Cin multiple of 16")
        if c.Cout < 8 or c.Cout % 8:
            bad.append("Cout multiple of 8")
        if s not in (1, 2) or kh * kw > 32 or not (0 <= ph < kh and 0 <= pw < kw):
            bad.append("kernel / stride / padding")
        if c.H + 2 * ph < kh or c.W + 2 * pw < kw or (s == 2 and min(c.H, c.W) < 2):
            bad.append("kernel larger than the padded map")
        if o["x_ctot"] % 8 or o["out_ctot"] % 8 or o["x_c0"] % 8 or o["out_c0"] % 8:
            bad.append("channel strides / offsets multiples of 8")
        if o["x_c0"] + c.Cin > o["x_ctot"] or o["out_c0"] + c.Cout > o["out_ctot"]:
            bad.append("channel slice outside the tensor")
        return bad
    if c.kind == CONV4S2 and (c.H | c.W) & 1:
        bad.append("conv4x4s2 needs even H, W")
    Wg, Hg = _grid(c)
    tile_grid = Wg >= 8 and Hg >= 16
    if c.entry in ("conv_fprop", "conv_dgrad"):
        K, N = (c.Cin, c.Cout) if c.entry == "conv_fprop" else (c.Cout, c.Cin)
        if K % 16 or N % 16:
            bad.append("K and N multiples of 16")
        split = o.get("splitk") or 1
        if not tile_grid or split > 1:
            if pick_tile(Wg, Hg, 128) is None:
                bad.append("gather grid must tile 128 pixels")
            bk = 64 if K % 64 == 0 else (32 if K % 32 == 0 else 16)
            if N in (160, 192) and bk == 16:
                bad.append("no 160 / 192-wide gather instance with BK = 16")
        if o.get("bias9") and (c.kind != CONV3 or not tile_grid or split > 1):
            bad.append("region bias needs a tile-resident 3x3 convolution")
        if o.get("stats") and o.get("act"):
            bad.append("fused activation excludes statistics")
        if o.get("groups", 1) > 1 and c.B % o["groups"]:
            bad.append("batch not divisible into statistics groups")
        return bad
    # conv_wgrad
    if c.Cin % 16 or c.Cout % 16:
        bad.append("Cin and Cout multiples of 16")
    on_tile = tile_grid and (c.Cout <= 128 or c.B * Wg * Hg >= 128 * 16 * 148)
    if not on_tile:
        if c.Cout % 32:
            bad.append("gather wgrad needs Cout % 32 == 0")
        if c.Cin > 16 and c.Cin % 32 == 16:
            bad.append("gather wgrad: no CWB = 16 instance for BN >= 64")
        if pick_tile(Wg, Hg, 64) is None:
            bad.append("gather wgrad grid must tile 64 pixels")
    return bad


# ---------------------------------------------------------------------------------------------- NaN poisoning
class NanTorch:
    """Stands in for the `torch` module inside sg2b200.ops: `empty` / `empty_like` return memory filled with NaN, so an
    output element (or split-K slab element) that a kernel fails to write reaches the checker as NaN, not as whatever
    the allocator left there. Everything else is torch itself."""

    def __init__(self, torch_module):
        self._torch = torch_module

    def __getattr__(self, name):
        return getattr(self._torch, name)

    @staticmethod
    def _poison(t):
        if t.is_floating_point():
            t.fill_(math.nan)
        return t

    def empty(self, *a, **k):
        return self._poison(self._torch.empty(*a, **k))

    def empty_like(self, *a, **k):
        return self._poison(self._torch.empty_like(*a, **k))
