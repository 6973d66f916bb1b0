"""GPU: the compute entry points of include/pv_b200.h, each compared with a float64 CPU reference of the same operation.

The model goldens reach most kernels only through whole networks, with bounds loose enough to hide a wrong edge tile,
padding row or stride.  Here every case:
  * uses operands on the f16 grid (f16 cases), so kernel and reference multiply identical values;
  * checks EVERY element against a bound scaled to that element (``tolerance``): f16 storage
    |d| <= 2^-10 |ref| + 1e-4 S + 1e-6, f32 |d| <= 1e-5 |ref| + 1e-5 S, where S is the sum of the absolute terms
    that make up the element (for a convolution |scale| conv(|x|, |w|) + |bias| (+ |residual|)).  One dropped tap
    moves an output by about S / taps, far outside the bound (tests/test_host_logic.py checks that on the CPU);
  * fills the buffers a direct ABI call writes with NaN first, then checks that the valid channels match, that pad
    lanes are exactly zero and that everything outside the written slice is still NaN;
  * asserts the route it took (plan statistics, host predicates and the names of the kernels that ran), so a shape
    change cannot silently move a case to another kernel.  Every case prints its route and worst error / bound.
"""
import ctypes as C
import functools
import math

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from pytorchvideo_b200 import _lib as L
from pytorchvideo_b200.engine import packing as PK
from pytorchvideo_b200.testing import f16_exact

pytestmark = pytest.mark.gpu

_DT = {"f16": L.PV_F16, "f32": L.PV_F32}
_TDT = {"f16": torch.float16, "f32": torch.float32}
_ACTS = {"none": L.ACT_NONE, "relu": L.ACT_RELU, "swish": L.ACT_SWISH, "gelu": L.ACT_GELU, "sigmoid": L.ACT_SIGMOID}


# ---------------------------------------------------------------------------------------------------------------
# float64 references and the per-element bound (also used by the CPU self-check in tests/test_host_logic.py)
# ---------------------------------------------------------------------------------------------------------------
def act_ref(y, act):
    if act in (None, "none"):
        return y
    if act == "relu":
        return torch.relu(y)
    if act == "swish":
        return y * torch.sigmoid(y)
    if act == "gelu":          # exact erf GELU
        return 0.5 * y * (1.0 + torch.erf(y / math.sqrt(2.0)))
    if act == "sigmoid":
        return torch.sigmoid(y)
    raise ValueError(act)


def conv_reference(x, w, scale, bias, stride, padding, dilation=(1, 1, 1), groups=1, act=None, res=None):
    """float64 act(conv3d(x, w) * scale + bias (+ res)) and S = |scale| conv3d(|x|, |w|) + |bias| (+ |res|)."""
    x64, w64 = x.double(), w.double()
    y = F.conv3d(x64, w64, None, stride, padding, dilation, groups)
    s_abs = F.conv3d(x64.abs(), w64.abs(), None, stride, padding, dilation, groups)
    sc = scale.double().view(1, -1, 1, 1, 1)
    b = bias.double().view(1, -1, 1, 1, 1)
    y = y * sc + b
    S = s_abs * sc.abs() + b.abs()
    if res is not None:
        y = y + res.double()
        S = S + res.double().abs()
    return act_ref(y, act), S


def tolerance(ref, S, dtype):
    """Per-element bound of an output stored as `dtype` (f16: one rounding of the stored value plus fp32
    accumulation; f32: fp32 accumulation)."""
    if dtype == "f16":
        return 2.0 ** -10 * ref.abs() + 1e-4 * S + 1e-6
    return 1e-5 * ref.abs() + 1e-5 * S


def worst_ratio(got, ref, S, dtype, extra=None):
    """max |got - ref| / bound over all elements (inf if any element is NaN)."""
    tol = tolerance(ref, S, dtype) + (0 if extra is None else extra)
    err = (got.double() - ref).abs()
    if bool(torch.isnan(err).any()):
        return float("inf")
    return float((err / tol).max())


def assert_close(got, ref, S, dtype, what, extra=None):
    assert got.shape == ref.shape, (got.shape, ref.shape)
    r = worst_ratio(got, ref, S, dtype, extra)
    err = float((got.double() - ref).abs().max())
    print("%s: max|d| = %.3e, worst |d| / bound = %.3f" % (what, err, r))
    if r > 1.0:
        flat = ((got.double() - ref).abs() / (tolerance(ref, S, dtype) + (0 if extra is None else extra))).reshape(-1)
        i = int(torch.nan_to_num(flat, nan=float("inf")).argmax())
        raise AssertionError("%s: element %d: kernel %r, reference %r, S %r (worst |d|/bound %.3f)"
                             % (what, i, float(got.reshape(-1)[i]), float(ref.reshape(-1)[i]),
                                float(S.reshape(-1)[i]), r))


# ---------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _nan(shape, dtype):
    return torch.full(shape, float("nan"), dtype=_TDT.get(dtype, dtype), device=_dev())


def _launched(fn):
    """Names of the CUDA kernels `fn` launches (torch.profiler), in launch order."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "kernel" in e.name and not e.name.startswith("cuda")]
    return names


def _assert_route(kernels, want, absent=()):
    for k in want:
        assert any(k in n for n in kernels), "expected kernel %s, launched %s" % (k, kernels)
    for k in absent:
        assert not any(k in n for n in kernels), "unexpected kernel %s, launched %s" % (k, kernels)
    print("route:", ", ".join(sorted(set(n.split("(")[0].split("<")[0].replace("void ", "") for n in kernels))))


def _rows(x_ncdhw, row_stride, off, dtype, fill=float("nan")):
    """[N,C,T,H,W] -> device [N*T*H*W, row_stride] with the C channels at [off, off + C) and `fill` elsewhere."""
    N, Cc = x_ncdhw.shape[:2]
    r = x_ncdhw.permute(0, 2, 3, 4, 1).reshape(-1, Cc)
    buf = torch.full((r.shape[0], row_stride), fill, dtype=_TDT[dtype])
    buf[:, off:off + Cc] = r.to(_TDT[dtype])
    return buf.to(_dev())


def _from_rows(rows, shape):
    """device [M, >= C] (valid channels first) -> CPU float64 [N, C, T, H, W]."""
    N, Cc, T, H, W = shape
    return rows[:, :Cc].double().cpu().reshape(N, T, H, W, Cc).permute(0, 4, 1, 2, 3)


def _folded_bn(co, seed):
    g = torch.Generator().manual_seed(seed)
    bn = nn.BatchNorm3d(co).eval()
    with torch.no_grad():
        bn.weight.copy_(torch.rand(co, generator=g) + 0.5)
        bn.bias.copy_(torch.rand(co, generator=g) - 0.5)
        bn.running_mean.copy_(torch.rand(co, generator=g) - 0.5)
        bn.running_var.copy_(torch.rand(co, generator=g) + 0.5)
    return bn


def _conv_operands(N, Ci, T, H, W, Co, k, seed, groups=1):
    g = torch.Generator().manual_seed(seed)
    x = f16_exact(torch.randn(N, Ci, T, H, W, generator=g))
    fan_in = Ci // groups * k[0] * k[1] * k[2]
    w = f16_exact(torch.randn(Co, Ci // groups, *k, generator=g) * (2.0 / fan_in) ** 0.5)
    return x, w


# ---------------------------------------------------------------------------------------------------------------
# A. Stem routes at the real model geometries, built the way ops.conv3d_bn_act builds them (lazy network input,
#    production route choice in Plan.emit_conv)
# ---------------------------------------------------------------------------------------------------------------
# name: (Co, kernel, stride, padding, conv bias instead of BN, T)
STEMS = {
    "x3d": (24, (1, 3, 3), (1, 2, 2), (0, 1, 1), False, 2),           # X3D conv_xy
    "slow": (64, (1, 7, 7), (1, 2, 2), (0, 3, 3), False, 2),          # Slow / C2D / R(2+1)D / detection
    "fast": (8, (5, 7, 7), (1, 2, 2), (2, 3, 3), False, 3),           # SlowFast Fast pathway: 40-channel taps GEMM
    "csn": (64, (3, 7, 7), (1, 2, 2), (1, 3, 3), False, 3),           # CSN: 192-channel taps GEMM
    "i3d": (64, (5, 7, 7), (1, 2, 2), (2, 3, 3), False, 3),           # I3D: 35 filter rows
    "i3d_co48": (48, (5, 7, 7), (1, 2, 2), (2, 3, 3), False, 3),      # widest taps GEMM: 5 x 48 = 240 channels
    "mvit": (96, (3, 7, 7), (2, 4, 4), (1, 3, 3), True, 3),           # MViT patch embed (bias, no BN), lead pixel
}
# production f16 route per stem: "stem_rows" | "taps" (taps GEMM on stem rows + tap sum) | "window" (window-mode igemm).
# I3D's 35 filter rows never reach the stem-rows kernel: with Co = 64 the packed weights (140 KiB) exceed its 120 KiB
# budget, and with Co <= 48 the kt * Co taps GEMM fits in 256 channels and is preferred.
STEM_ROUTE = {"x3d": "stem_rows", "slow": "stem_rows", "fast": "taps", "csn": "taps", "i3d": "window",
              "i3d_co48": "taps", "mvit": "window"}
# (stem, H, W, clip dtype)
STEM_GEOMS = [
    ("x3d", 160, 160, "f32"), ("x3d", 224, 224, "f32"), ("x3d", 312, 312, "f32"),     # 312: Wo = 156, two W tiles
    ("x3d", 160, 158, "f32"),                                                          # W % 4 != 0
    ("x3d", 160, 160, "f16"),                                                          # f16 host clip
    ("slow", 224, 224, "f32"), ("slow", 224, 222, "f32"), ("slow", 224, 224, "f16"),
    ("fast", 224, 224, "f32"), ("csn", 224, 224, "f32"), ("i3d", 224, 224, "f32"), ("i3d_co48", 224, 224, "f32"),
    ("mvit", 224, 224, "f32"), ("mvit", 112, 112, "f32"), ("mvit", 112, 112, "f16"),
]
STEM_MODES = ["f16", "f16_no_stem_rows", "f32"]


@functools.lru_cache(maxsize=None)
def _stem_problem(stem, H, W, clip):
    """Operands + float64 reference of one stem geometry (N = 2), shared by the three modes."""
    Co, k, s, p, use_bias, T = STEMS[stem]
    x, w = _conv_operands(2, 3, T, H, W, Co, k, seed=H + W + Co + k[0])
    if use_bias:
        conv_bias, bn = f16_exact(torch.rand(Co, generator=torch.Generator().manual_seed(3)) * 0.2 - 0.1), None
    else:
        conv_bias, bn = None, _folded_bn(Co, 11)
    scale, bias = PK.fold_bn(conv_bias, bn, Co, Co)
    ref, S = conv_reference(x, w, scale, bias, s, p, act="relu")
    # taps route: the per-tap partial sums are stored in f16 once (pv_temporal_tap_sum): add that one rounding
    wt =torch.cat([w[:, :, j:j + 1] for j in range(k[0])], 0)
    yk = F.conv3d(x.double(), wt.double(), None, (1, s[1], s[2]), (0, p[1], p[2])).abs()
    To = ref.shape[2]
    part = torch.zeros_like(ref)
    for t in range(To):
        for j in range(k[0]):
            ti = t * s[0] + j - p[0]
            if 0 <= ti < T:
                part[:, :, t] += yk[:, j * Co:(j + 1) * Co, ti]
    taps_extra = 2.0 ** -11 * part * scale.double().abs().view(1, -1, 1, 1, 1)
    return x if clip == "f32" else x.half(), w, conv_bias, bn, ref, S, taps_extra


def _run_plan_conv(x, w, conv_bias, bn, stride, padding, act, dtype):
    from pytorchvideo_b200.engine.plan import Plan
    plan = Plan(_dev(), _DT[dtype], use_tcgen05=True)
    xin = x.to(_dev()).contiguous()
    cin = x.shape[1]
    xr = plan.emit_input_ncdhw(xin, cin, 4 if cin <= 4 else PK.pad8(cin))
    y = plan.emit_conv(xr, w, conv_bias, bn, stride, padding, (1, 1, 1), 1, _ACTS[act], None, "stem")
    out, shape = plan.emit_to_ncdhw(y)
    plan.finalize()
    kernels = _launched(lambda: plan.run(_stream()))
    n = math.prod(shape)
    return out.tensor[:n].view(*shape).double().cpu(), plan, kernels


@pytest.mark.parametrize("mode", STEM_MODES)
@pytest.mark.parametrize("stem,H,W,clip", STEM_GEOMS,
                         ids=["%s-%dx%d-%sclip-%s" % (g[0], g[1], g[2], g[3], STEM_ROUTE[g[0]]) for g in STEM_GEOMS])
def test_stem_routes(stem, H, W, clip, mode, monkeypatch):
    """Stem convolutions through pv_conv3d_stem_rows_fwd, window-mode pv_conv3d_fwd or the factored taps GEMM +
    pv_temporal_tap_sum, fed by pv_ncdhw_to_ndhwc_padw (4-pixel f32 kernel or the generic one); f32 parity mode takes
    pv_ncdhw_to_ndhwc + the direct kernel."""
    Co, k, s, p, _, T = STEMS[stem]
    x, w, conv_bias, bn, ref, S, taps_extra = _stem_problem(stem, H, W, clip)
    if mode == "f16_no_stem_rows":
        monkeypatch.setenv("PVB200_NO_STEMROWS", "1")
    dtype = "f32" if mode == "f32" else "f16"
    got, plan, kernels = _run_plan_conv(x, w, conv_bias, bn, s, p, "relu", dtype)
    names = [m["name"] for m in plan.meta]
    route = STEM_ROUTE[stem]
    if dtype == "f32":
        assert names == ["ncdhw_to_ndhwc", "stem", "to_ncdhw"] and plan.stats["direct"] == 1
        _assert_route(kernels, ["ncdhw_to_ndhwc_kernel", "conv3d_direct_kernel"], ["igemm", "stem_rows"])
    else:
        four_px = clip == "f32" and W % 4 == 0
        conv_kernel = "conv3d_stem_rows_kernel" if mode == "f16" and route != "window" else "conv3d_igemm_kernel"
        if route == "taps":
            assert names == ["ncdhw_to_ndhwc_padw", "stem.taps", "stem.tapsum", "to_ncdhw"], names
            want = [conv_kernel, "temporal_tap_sum_kernel"]
        else:
            assert names == ["ncdhw_to_ndhwc_padw", "stem", "to_ncdhw"], names
            want = [conv_kernel]
        assert plan.stats.get("stem_rows", 0) == (1 if "stem_rows" in conv_kernel else 0)
        want.append("ncdhw_f32_to_ndhwc4_padw_kernel" if four_px else "ncdhw_to_ndhwc_padw_kernel")
        _assert_route(kernels, want, ["conv3d_direct_kernel", "gather"] +
                      (["ncdhw_f32_to_ndhwc4_padw_kernel"] if not four_px else []))
    extra = taps_extra if (route == "taps" and dtype == "f16") else None
    assert_close(got, ref, S, dtype, "%s %dx%d %s clip, %s" % (stem, H, W, clip, mode), extra)


# ---------------------------------------------------------------------------------------------------------------
# B. Layout conversions: copies plus at most one rounding -> bit equality, NaN canaries, zero pad lanes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src_dt,dst_dt", [("f32", "f16"), ("f32", "f32"), ("f16", "f16"), ("f16", "f32")])
def test_ncdhw_to_ndhwc(src_dt, dst_dt):
    lib = L.load()
    N, Cc, T, H, W, c_pad, rs = 2, 5, 3, 7, 9, 8, 12          # pad lanes [5, 8), canaries [8, 12)
    src = torch.randn(N, Cc, T, H, W, generator=torch.Generator().manual_seed(1)).to(_TDT[src_dt])
    srcd = src.to(_dev())
    M = N * T * H * W
    dst = _nan((M + 3, rs), dst_dt)                            # three canary rows past the end
    kernels = _launched(lambda: L.check(lib.pv_ncdhw_to_ndhwc(srcd.data_ptr(), _DT[src_dt], dst.data_ptr(), _DT[dst_dt], N, Cc,
                                                              T, H, W, c_pad, rs, _stream()), "pv_ncdhw_to_ndhwc"))
    _assert_route(kernels, ["ncdhw_to_ndhwc_kernel"])
    got = dst.cpu()
    want = src.permute(0, 2, 3, 4, 1).reshape(M, Cc).to(_TDT[dst_dt])
    assert torch.equal(got[:M, :Cc], want)
    assert bool((got[:M, Cc:c_pad] == 0).all())
    assert bool(torch.isnan(got[:M, c_pad:]).all()) and bool(torch.isnan(got[M:]).all())


# (src dtype, dst dtype, W, source offset in elements) -> kernel
PADW_CASES = [
    ("f32", "f16", 16, 0, "ncdhw_f32_to_ndhwc4_padw_kernel"),
    ("f32", "f16", 18, 0, "ncdhw_to_ndhwc_padw_kernel"),     # W % 4 != 0
    ("f32", "f16", 16, 1, "ncdhw_to_ndhwc_padw_kernel"),     # source not 16-byte aligned
    ("f16", "f16", 16, 0, "ncdhw_to_ndhwc_padw_kernel"),     # f16 host clip
    ("f32", "f32", 16, 0, "ncdhw_to_ndhwc_padw_kernel"),
]


@pytest.mark.parametrize("src_dt,dst_dt,W,off,kernel", PADW_CASES,
                         ids=["%s-%s-W%d-off%d-%s" % (c[0], c[1], c[2], c[3], "4px" if "4_padw" in c[4] else "generic")
                              for c in PADW_CASES])
def test_ncdhw_to_ndhwc_padw(src_dt, dst_dt, W, off, kernel):
    lib = L.load()
    N, Cc, T, H, c_pad, w_pad = 2, 3, 2, 5, 4, 4
    w_phys = (w_pad + W + 3 + 3) // 4 * 4                      # zeros on the right as well
    src = torch.randn(N, Cc, T, H, W, generator=torch.Generator().manual_seed(2)).to(_TDT[src_dt])
    flat = torch.empty(src.numel() + 8, dtype=src.dtype)
    flat[off:off + src.numel()] = src.reshape(-1)
    srcd = flat.to(_dev())
    M = N * T * H * w_phys
    tail = 8 * c_pad                                           # the caller's slack past the rows: never written
    dst = _nan((M * c_pad + tail,), dst_dt)
    esz = src.element_size()
    kernels = _launched(lambda: L.check(lib.pv_ncdhw_to_ndhwc_padw(srcd.data_ptr() + off * esz, _DT[src_dt], dst.data_ptr(),
                                                                   _DT[dst_dt], N, Cc, T, H, W, c_pad, w_pad, w_phys,
                                                                   _stream()), "pv_ncdhw_to_ndhwc_padw"))
    _assert_route(kernels, [kernel])
    got = dst.cpu()
    rows = got[:M * c_pad].view(N, T, H, w_phys, c_pad)
    want = torch.zeros(N, T, H, w_phys, c_pad, dtype=_TDT[dst_dt])
    want[:, :, :, w_pad:w_pad + W, :Cc] = src.permute(0, 2, 3, 4, 1).to(_TDT[dst_dt])
    assert torch.equal(rows, want)                             # values, zero pad pixels and zero pad lanes
    assert bool(torch.isnan(got[M * c_pad:]).all())


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_ndhwc_to_ncdhw_strided(dt):
    lib = L.load()
    N, Cc, T, H, W, rs = 2, 12, 3, 5, 7, 24
    src = torch.randn(N * T * H * W, rs, generator=torch.Generator().manual_seed(3)).to(_TDT[dt])
    src[:, Cc:] = float("nan")                                 # channels past C must never be read
    total = N * Cc * T * H * W
    dst = _nan((total + 16,), torch.float32)
    srcd = src.to(_dev())
    kernels = _launched(lambda: L.check(lib.pv_ndhwc_to_ncdhw(srcd.data_ptr(), _DT[dt], rs, dst.data_ptr(), N, Cc, T, H, W,
                                                              _stream()), "pv_ndhwc_to_ncdhw"))
    _assert_route(kernels, ["ndhwc_to_ncdhw_kernel"])
    got = dst.cpu()
    want = src[:, :Cc].float().reshape(N, T, H, W, Cc).permute(0, 4, 1, 2, 3).reshape(-1)
    assert torch.equal(got[:total], want)
    assert bool(torch.isnan(got[total:]).all())


# ---------------------------------------------------------------------------------------------------------------
# C. Convolution ABI edges: pv_conv3d_fwd / pv_dwconv3d_fwd called directly with engine/packing.py weights
# ---------------------------------------------------------------------------------------------------------------
def _conv_abi(x, w, scale, bias, stride, pad, dil, *, path, dtype, act="none", res=None, x_rs=None, x_off=0,
              y_rs=None, y_off=0, r_rs=None, depthwise=False):
    """Run one convolution through the ABI on NDHWC buffers with channel slices.  Returns (y rows [M, y_rs] on the
    CPU, launched kernel names).  path: "tcgen05" | "direct" | "depthwise"."""
    lib = L.load()
    N, Ci, T, H, W = x.shape
    Co = w.shape[0]
    co_pad = PK.pad8(Co)
    k = tuple(w.shape[2:])
    To, Ho, Wo = [(i + 2 * p_ - d_ * (k_ - 1) - 1) // s_ + 1 for i, k_, s_, p_, d_ in zip((T, H, W), k, stride, pad, dil)]
    x_rs = x_rs or Ci
    y_rs = y_rs or co_pad
    tdt = _TDT[dtype]
    xb = _rows(x, x_rs, x_off, dtype)
    M = N * To * Ho * Wo
    yb = _nan((M, y_rs), dtype)
    rb = None
    if res is not None:
        r_rs = r_rs or co_pad
        rfull = torch.zeros(N, co_pad, To, Ho, Wo)
        rfull[:, :Co] = res
        rb = _rows(rfull, r_rs, 0, dtype)
    sc = torch.zeros(co_pad)
    bi = torch.zeros(co_pad)
    sc[:Co], bi[:Co] = scale, bias
    sc, bi = sc.to(_dev()), bi.to(_dev())
    d = L.Conv3dDesc()
    d.dtype = _DT[dtype]
    d.N, d.Ti, d.Hi, d.Wi, d.Ci = N, T, H, W, Ci
    d.To, d.Ho, d.Wo, d.Co = To, Ho, Wo, co_pad
    d.kt, d.kh, d.kw = k
    d.st, d.sh, d.sw = stride
    d.pt, d.ph, d.pw = pad
    d.dt, d.dh, d.dw = dil
    d.groups = Ci if depthwise else 1
    d.act = _ACTS[act]
    d.has_residual = 1 if res is not None else 0
    d.x_row_stride, d.y_row_stride, d.res_row_stride = x_rs, y_rs, (r_rs or 0)
    d.ci_pad64 = Ci if Ci < 64 else PK.pad_to(Ci, 64)
    esz = 2 if dtype == "f16" else 4
    xp, yp = xb.data_ptr() + x_off * esz, yb.data_ptr() + y_off * esz
    if depthwise:
        assert co_pad == Ci
        wd = PK.pack_depthwise(w, Ci, tdt).to(_dev())
        fn = lambda: L.check(lib.pv_dwconv3d_fwd(C.byref(d), xp, wd.data_ptr(), sc.data_ptr(), bi.data_ptr(), yp, None,
                                                 _stream()), "pv_dwconv3d_fwd")
    else:
        if path == "tcgen05":
            assert lib.pv_conv3d_tcgen05_supported(C.byref(d)) == 1
            wd = PK.pack_dense_tcgen05(w, d.ci_pad64, co_pad).to(_dev())
            algo = L.ALGO_TCGEN05
        else:
            wd = PK.pack_dense_direct(w, Ci, co_pad, tdt).to(_dev())
            algo = L.ALGO_DIRECT
        fn = lambda: L.check(lib.pv_conv3d_fwd(C.byref(d), algo, xp, wd.data_ptr(), sc.data_ptr(), bi.data_ptr(),
                                               rb.data_ptr() if rb is not None else None, yp, _stream()), "pv_conv3d_fwd")
    kernels = _launched(fn)
    return yb.cpu(), kernels, (N, Co, To, Ho, Wo)


def _check_conv_slice(yrows, shape, co_pad, y_off, ref, S, dtype, what):
    """valid channels vs the reference, pad lanes exactly 0, every other channel of the row still NaN."""
    Co = shape[1]
    got = _from_rows(yrows[:, y_off:], shape)
    assert_close(got, ref, S, dtype, what)
    assert bool((yrows[:, y_off + Co:y_off + co_pad] == 0).all()), "pad lanes not zero"
    assert bool(torch.isnan(yrows[:, :y_off]).all()) and bool(torch.isnan(yrows[:, y_off + co_pad:]).all()), \
        "write outside the output slice"


def _kernel_of(path, Ci):
    """Dense kernel the dispatcher must pick (pv_api.cu): C_in < 64 goes through the gather-fed kernel except the
    narrow TMA widths 16 / 32."""
    if path == "direct":
        return "conv3d_direct_kernel"
    return "conv3d_igemm_gather_kernel" if Ci < 64 and Ci not in (16, 32) else "conv3d_igemm_kernel"


# (Ci, path, dtype, kernel, dilation, padding), stride 1
DIL_CASES = [
    (512, "tcgen05", "f16", (1, 3, 3), (1, 2, 2), (0, 2, 2)),     # TMA-fed
    (32, "tcgen05", "f16", (1, 3, 3), (1, 2, 2), (0, 2, 2)),      # narrow TMA
    (24, "tcgen05", "f16", (1, 3, 3), (1, 2, 2), (0, 2, 2)),      # gather
    (48, "tcgen05", "f16", (1, 3, 3), (1, 2, 2), (0, 2, 2)),      # gather
    (24, "direct", "f16", (1, 3, 3), (1, 2, 2), (0, 2, 2)),
    (32, "direct", "f32", (1, 3, 3), (1, 2, 2), (0, 2, 2)),
    (64, "tcgen05", "f16", (3, 1, 1), (2, 1, 1), (2, 0, 0)),      # temporal dilation
    (64, "direct", "f32", (3, 1, 1), (2, 1, 1), (2, 0, 0)),
]


@pytest.mark.parametrize("Ci,path,dtype,k,dil,pad", DIL_CASES,
                         ids=["ci%d-%s-%s-k%s-dil%s-%s" % (c[0], c[1], c[2], "".join(map(str, c[3])), "".join(map(str, c[4])),
                                                          _kernel_of(c[1], c[0]).replace("conv3d_", "").replace("_kernel", ""))
                              for c in DIL_CASES])
def test_conv_dilation(Ci, path, dtype, k, dil, pad):
    """Dilated convolutions (detection trunks run res5 with dilation (1, 2, 2) on the tensor cores)."""
    N, T, H, W, Co = 2, 6, 11, 13, 60                          # Co 60 -> 64: four pad lanes
    x, w = _conv_operands(N, Ci, T, H, W, Co, k, seed=Ci + sum(dil))
    bn = _folded_bn(Co, 5)
    scale, bias = PK.fold_bn(None, bn, Co, Co)
    ref, S = conv_reference(x, w, scale, bias, (1, 1, 1), pad, dil, act="relu")
    y, kernels, shape = _conv_abi(x, w, scale, bias, (1, 1, 1), pad, dil, path=path, dtype=dtype, act="relu")
    _assert_route(kernels, [_kernel_of(path, Ci)])
    _check_conv_slice(y, shape, 64, 0, ref, S, dtype, "dilation %s Ci %d %s %s" % (dil, Ci, path, dtype))


# (C, kernel, stride, padding, dilation, dtype, kernel name)
DW_DIL_CASES = [
    (64, (3, 3, 3), (1, 1, 1), (2, 2, 1), (2, 2, 1), "f16", "dwconv3d_tile_kernel"),      # dt / dh dilation: TMA stencil
    (64, (1, 3, 3), (1, 1, 1), (0, 1, 2), (1, 1, 2), "f16", "dwconv3d_kernel"),           # dw dilation: generic stencil
    (64, (1, 3, 3), (1, 1, 1), (0, 1, 2), (1, 1, 2), "f32", "dwconv3d_kernel"),
    (48, (3, 3, 3), (1, 2, 2), (2, 1, 1), (2, 1, 1), "f32", "dwconv3d_w4_kernel"),
]


@pytest.mark.parametrize("Cc,k,s,pad,dil,dtype,kernel", DW_DIL_CASES,
                         ids=["c%d-dil%s-%s-%s" % (c[0], "".join(map(str, c[4])), c[5], c[6].replace("_kernel", ""))
                              for c in DW_DIL_CASES])
def test_dwconv_dilation(Cc, k, s, pad, dil, dtype, kernel):
    N, T, H, W = 2, 6, 12, 14
    x, w = _conv_operands(N, Cc, T, H, W, Cc, k, seed=Cc + sum(dil), groups=Cc)
    bn = _folded_bn(Cc, 6)
    scale, bias = PK.fold_bn(None, bn, Cc, Cc)
    ref, S = conv_reference(x, w, scale, bias, s, pad, dil, groups=Cc, act="swish")
    y, kernels, shape = _conv_abi(x, w, scale, bias, s, pad, dil, path="depthwise", dtype=dtype, act="swish",
                                  y_rs=Cc + 16, y_off=8, depthwise=True)
    _assert_route(kernels, [kernel])
    _check_conv_slice(y, shape, Cc, 8, ref, S, dtype, "depthwise dilation %s %s" % (dil, dtype))


# (Ci, path, dtype): the input is channels [8, 8 + Ci) of a wider buffer, the output goes to channels [8, 8 + Co_pad)
# of another one, the residual has its own row stride; every neighbouring channel holds NaN
SLICE_CASES = [(64, "tcgen05", "f16"), (32, "tcgen05", "f16"), (16, "tcgen05", "f16"), (24, "tcgen05", "f16"),
               (24, "direct", "f16"), (24, "direct", "f32")]


@pytest.mark.parametrize("Ci,path,dtype", SLICE_CASES,
                         ids=["ci%d-%s-%s-%s" % (c[0], c[1], c[2], _kernel_of(c[1], c[0]).replace("conv3d_", "")
                                                                   .replace("_kernel", "")) for c in SLICE_CASES])
def test_conv_channel_slices(Ci, path, dtype):
    """torch.cat fused away: x_row_stride > Ci, y_row_stride > Co, res_row_stride of its own."""
    N, T, H, W, Co = 2, 3, 9, 11, 44                           # Co 44 -> 48
    k, s, p = (1, 3, 3), (1, 2, 2), (0, 1, 1)
    x, w = _conv_operands(N, Ci, T, H, W, Co, k, seed=Ci + 7)
    bn = _folded_bn(Co, 8)
    scale, bias = PK.fold_bn(None, bn, Co, Co)
    To, Ho, Wo = T, (H - 1) // 2 + 1, (W - 1) // 2 + 1
    res = f16_exact(torch.randn(N, Co, To, Ho, Wo, generator=torch.Generator().manual_seed(9)))
    ref, S = conv_reference(x, w, scale, bias, s, p, act="relu", res=res)
    y, kernels, shape = _conv_abi(x, w, scale, bias, s, p, (1, 1, 1), path=path, dtype=dtype, act="relu", res=res,
                                  x_rs=Ci + 16, x_off=8, y_rs=48 + 24, y_off=8, r_rs=48 + 8)
    _assert_route(kernels, [_kernel_of(path, Ci)])
    _check_conv_slice(y, shape, 48, 8, ref, S, dtype, "channel slices Ci %d %s %s" % (Ci, path, dtype))


@pytest.mark.parametrize("Co", [96, 192])
def test_conv_residual_ring_x3d_widths(Co):
    """Pointwise conv + residual at X3D widths with >= 3 tiles per CTA on 148 SMs (the staging ring wraps): Co 96 ends
    in half of a 64-channel staging sub-tile, Co 192 runs three sub-tiles through the single-team ring."""
    N, T, H, W, Ci = 1, 4, 128, 128, 64
    x, w = _conv_operands(N, Ci, T, H, W, Co, (1, 1, 1), seed=Co)
    bn = _folded_bn(Co, 9)
    scale, bias = PK.fold_bn(None, bn, Co, Co)
    res = f16_exact(torch.randn(N, Co, T, H, W, generator=torch.Generator().manual_seed(10)))
    ref, S = conv_reference(x, w, scale, bias, (1, 1, 1), (0, 0, 0), act="relu", res=res)
    y, kernels, shape = _conv_abi(x, w, scale, bias, (1, 1, 1), (0, 0, 0), (1, 1, 1), path="tcgen05", dtype="f16",
                                  act="relu", res=res, y_rs=Co + 16, y_off=8, r_rs=Co + 8)
    _assert_route(kernels, ["conv3d_igemm_kernel"])
    _check_conv_slice(y, shape, Co, 8, ref, S, "f16", "residual ring Co %d" % Co)


@pytest.mark.parametrize("dtype", ["f16", "f32"])
def test_temporal_tap_sum_strided(dtype):
    """pv_temporal_tap_sum with temporal stride, dilation and both padding edges; input rows wider than kt*Co and
    output rows wider than Co (the neighbouring channels hold NaN)."""
    lib = L.load()
    N, Ti, hw, Co, kt, st, pt, dil = 2, 7, 37, 16, 3, 2, 2, 2
    To = (Ti + 2 * pt - dil * (kt - 1) - 1) // st + 1
    irs, ors = kt * Co + 8, Co + 8
    g = torch.Generator().manual_seed(12)
    yk = f16_exact(torch.randn(N, Ti, hw, kt * Co, generator=g))
    scale, bias = torch.rand(Co, generator=g) + 0.5, torch.rand(Co, generator=g) - 0.5
    ykb = torch.full((N * Ti * hw, irs), float("nan"), dtype=_TDT[dtype])
    ykb[:, :kt * Co] = yk.reshape(-1, kt * Co).to(_TDT[dtype])
    ykb = ykb.to(_dev())
    y = _nan((N * To * hw, ors), dtype)
    sd, bd = scale.to(_dev()), bias.to(_dev())
    kernels = _launched(lambda: L.check(lib.pv_temporal_tap_sum(ykb.data_ptr(), y.data_ptr(), _DT[dtype], N, Ti, To, hw, Co, kt, st,
                                                                pt, dil, sd.data_ptr(), bd.data_ptr(), L.ACT_GELU, irs, ors,
                                                                _stream()), "pv_temporal_tap_sum"))
    _assert_route(kernels, ["temporal_tap_sum_kernel"])
    acc = torch.zeros(N, To, hw, Co, dtype=torch.float64)
    sab = torch.zeros_like(acc)
    for t in range(To):
        for j in range(kt):
            ti = t * st + j * dil - pt
            if 0 <= ti < Ti:
                acc[:, t] += yk[:, ti, :, j * Co:(j + 1) * Co].double()
                sab[:, t] += yk[:, ti, :, j * Co:(j + 1) * Co].double().abs()
    pre = acc * scale.double() + bias.double()
    ref = act_ref(pre, "gelu")
    S = sab * scale.double() + bias.double().abs()
    got = y.cpu()
    assert_close(got[:, :Co].double().reshape(ref.shape), ref, S, dtype, "temporal tap sum %s" % dtype)
    assert bool(torch.isnan(got[:, Co:]).all())


# ---------------------------------------------------------------------------------------------------------------
# D. Token kernels as the engine calls them
# ---------------------------------------------------------------------------------------------------------------
ATT_KERNEL = {"tc": "attention_tc_kernel", "mma": "attention_mma_kernel", "simt": "attention_kernel"}
# (path, dtype, B, heads, D, Nq, Nk, residual, o row padding, logit amplitude); Nq == Nk: q|k|v slices of ONE
# [B, N, 3 dim] buffer (engine/plan.py emit_attention); else q has its own buffer and k|v share one
ATT_CASES = [
    ("tc", "f16", 2, 2, 32, 50, 50, False, 0, 1.0),
    ("tc", "f16", 2, 2, 64, 50, 50, True, 0, 1.0),
    ("tc", "f16", 1, 2, 96, 197, 197, True, 0, 1.0),
    ("tc", "f16", 2, 1, 64, 1, 1, False, 0, 1.0),
    ("tc", "f16", 2, 2, 64, 1, 129, False, 0, 1.0),
    ("tc", "f16", 2, 2, 96, 37, 129, True, 0, 1.0),
    ("tc", "f16", 2, 2, 64, 65, 65, False, 0, 7.0),        # logits ~ +-50: the two-sweep max
    ("mma", "f16", 2, 1, 128, 50, 50, False, 0, 1.0),
    ("mma", "f16", 2, 2, 128, 1, 129, True, 0, 1.0),
    ("mma", "f16", 2, 2, 64, 50, 50, True, 2, 1.0),         # o_row_stride = 130 = 2 (mod 8): TMA path declines
    ("simt", "f32", 2, 2, 32, 50, 50, False, 0, 1.0),
    ("simt", "f32", 2, 2, 64, 33, 129, True, 0, 1.0),
    ("simt", "f32", 2, 1, 128, 50, 50, False, 0, 1.0),
    ("simt", "f32", 2, 2, 64, 65, 65, False, 0, 7.0),
]


@pytest.mark.parametrize("path,dtype,B,heads,D,Nq,Nk,resid,o_pad,amp", ATT_CASES,
                         ids=["%s-%s-D%d-q%d-k%d%s%s%s" % (c[0], c[1], c[4], c[5], c[6], "-resid" if c[7] else "",
                                                          "-ors%d" % (c[3] * c[4] + c[8]) if c[8] else "",
                                                          "-logits50" if c[9] > 1 else "") for c in ATT_CASES])
def test_attention_as_the_engine_calls_it(path, dtype, B, heads, D, Nq, Nk, resid, o_pad, amp):
    lib = L.load()
    dim = heads * D
    g = torch.Generator().manual_seed(D + Nq + Nk)
    tdt = _TDT[dtype]
    scale = D ** -0.5
    if Nq == Nk:
        buf = torch.randn(B, Nk, 3 * dim, generator=g)
        buf[..., :2 * dim] *= amp
        buf = f16_exact(buf)
        q, k, v = buf[..., :dim], buf[..., dim:2 * dim], buf[..., 2 * dim:]
        qb = kb = buf.to(tdt).to(_dev())
        q_off, k_off, v_off, q_rs, kv_rs = 0, dim, 2 * dim, 3 * dim, 3 * dim
    else:
        qh = f16_exact(torch.randn(B, Nq, dim, generator=g) * amp)
        kvh = torch.randn(B, Nk, 2 * dim, generator=g)
        kvh[..., :dim] *= amp
        kvh = f16_exact(kvh)
        q, k, v = qh, kvh[..., :dim], kvh[..., dim:]
        qb, kb = qh.to(tdt).to(_dev()), kvh.to(tdt).to(_dev())
        q_off, k_off, v_off, q_rs, kv_rs = 0, 0, dim, dim, 2 * dim
    o_rs = dim + o_pad
    o = _nan((B * Nq * o_rs + 8,), dtype)
    d = L.AttentionDesc()
    d.dtype, d.B, d.H, d.Nq, d.Nk, d.D = _DT[dtype], B, heads, Nq, Nk, D
    d.q_row_stride, d.k_row_stride, d.v_row_stride, d.o_row_stride = q_rs, kv_rs, kv_rs, o_rs
    d.q_batch_stride, d.k_batch_stride, d.v_batch_stride, d.o_batch_stride = Nq * q_rs, Nk * kv_rs, Nk * kv_rs, Nq * o_rs
    d.scale, d.add_q_residual = float(scale), 1 if resid else 0
    esz = 2 if dtype == "f16" else 4
    kernels = _launched(lambda: L.check(lib.pv_attention_fwd(C.byref(d), qb.data_ptr() + q_off * esz, kb.data_ptr() + k_off * esz,
                                                             kb.data_ptr() + v_off * esz, o.data_ptr(), _stream()),
                                        "pv_attention_fwd"))
    _assert_route(kernels, [ATT_KERNEL[path]], [n for p_, n in ATT_KERNEL.items() if p_ != path])
    q4, k4, v4 = (t.double().reshape(B, -1, heads, D).transpose(1, 2) for t in (q, k, v))
    p = torch.softmax((q4 @ k4.transpose(-1, -2)) * scale, -1)
    ref = p @ v4
    S = p @ v4.abs()
    if resid:
        ref, S = ref + q4, S + q4.abs()
    # fp32 logits carry a rounding of their own absolute sum sum_i |q_i k_i| * scale, which the exponential turns into a
    # relative error of the probabilities: large (~ +-50) logits get a correspondingly wider bound
    lmax = ((q4.abs() @ k4.abs().transpose(-1, -2)) * scale).amax(-1, keepdim=True)
    logit_err = 2.0 ** -22 * lmax * S
    ref, S, logit_err = (t.transpose(1, 2).reshape(B, Nq, dim) for t in (ref, S, logit_err))
    got = o.cpu()
    rows = got[:B * Nq * o_rs].view(B * Nq, o_rs)
    # tensor-core paths round the probabilities to f16 for the P.V product (and normalise by the sum of the rounded
    # values): each weight carries a relative error up to 2^-10, hence the 2^-10 S term on top of the f16 bound
    extra = logit_err + (2.0 ** -10 * S if dtype == "f16" else 0)
    assert_close(rows[:, :dim].reshape(B, Nq, dim), ref, S, dtype, "attention %s D %d Nq %d Nk %d" % (path, D, Nq, Nk), extra)
    assert bool(torch.isnan(rows[:, dim:]).all()) and bool(torch.isnan(got[B * Nq * o_rs:]).all())


@pytest.mark.parametrize("x_dt,y_dt,fn", [("f16", "f16", "pv_add_pos_cls"), ("f32", "f32", "pv_add_pos_cls"),
                                          ("f16", "f32", "pv_add_pos_cls_to"), ("f16", "f16", "pv_add_pos_cls_to")])
@pytest.mark.parametrize("has_cls", [0, 1])
def test_add_pos_cls(x_dt, y_dt, fn, has_cls):
    lib = L.load()
    B, n_patch, Cc, x_rs = 2, 21, 48, 64
    g = torch.Generator().manual_seed(13)
    x = f16_exact(torch.randn(B, n_patch, x_rs, generator=g))
    x[..., Cc:] = float("nan")                                 # the rest of the wider source row is never read
    pos = torch.randn(n_patch + has_cls, Cc, generator=g) * 0.2
    xd, posd = x.to(_TDT[x_dt]).to(_dev()), pos.to(_dev())
    n_out = B * (n_patch + has_cls) * Cc
    y = _nan((n_out + 8,), y_dt)
    if fn == "pv_add_pos_cls":
        call = lambda: L.check(lib.pv_add_pos_cls(xd.data_ptr(), y.data_ptr(), _DT[x_dt], B, n_patch, Cc, x_rs, posd.data_ptr(),
                                                  has_cls, _stream()), fn)
    else:
        call = lambda: L.check(lib.pv_add_pos_cls_to(xd.data_ptr(), _DT[x_dt], y.data_ptr(), _DT[y_dt], B, n_patch, Cc, x_rs,
                                                     posd.data_ptr(), has_cls, _stream()), fn)
    _assert_route(_launched(call), ["add_pos_cls_kernel"])
    ref = torch.zeros(B, n_patch + has_cls, Cc, dtype=torch.float64)
    S = torch.zeros_like(ref)
    if has_cls:
        ref[:, 0], S[:, 0] = pos[0].double(), pos[0].double().abs()
    ref[:, has_cls:] = x[..., :Cc].double() + pos[has_cls:].double()
    S[:, has_cls:] = x[..., :Cc].double().abs() + pos[has_cls:].double().abs()
    got = y.cpu()
    assert_close(got[:n_out].view(ref.shape), ref, S, y_dt, "%s has_cls %d %s->%s" % (fn, has_cls, x_dt, y_dt))
    assert bool(torch.isnan(got[n_out:]).all())


@pytest.mark.parametrize("dtype", ["f16", "f32"])
def test_copy_rows_strided(dtype):
    lib = L.load()
    rows, Cc, s_rs, d_rs = 37, 48, 64, 56
    src = torch.randn(rows, s_rs, generator=torch.Generator().manual_seed(14)).to(_TDT[dtype])
    srcd = src.to(_dev())
    dst = _nan((rows + 1, d_rs), dtype)
    _assert_route(_launched(lambda: L.check(lib.pv_copy_rows(srcd.data_ptr(), dst.data_ptr(), _DT[dtype], rows, Cc, s_rs, d_rs,
                                                             _stream()), "pv_copy_rows")), ["copy_rows_kernel"])
    got = dst.cpu()
    assert torch.equal(got[:rows, :Cc], src[:, :Cc])
    assert bool(torch.isnan(got[:rows, Cc:]).all()) and bool(torch.isnan(got[rows:]).all())


@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("mode,k,s,p", [("max", (3, 3, 3), (1, 2, 2), (1, 1, 1)), ("max", (1, 3, 3), (1, 4, 4), (0, 1, 1)),
                                        ("avg", (3, 3, 3), (2, 2, 2), (1, 1, 1))])
def test_pool3d_token_batch_strides(mode, k, s, p, dtype):
    """MViT pool_skip: pooling over the patch tokens of [B, 1 + T*H*W, C] token tensors, stepping over the cls row of
    every sample with x_batch_stride / y_batch_stride; cls rows and the rest of each row stay untouched."""
    lib = L.load()
    B, T, H, W, Cc, x_rs, y_rs = 2, 4, 9, 10, 48, 56, 64
    To, Ho, Wo = [(i + 2 * p_ - k_) // s_ + 1 for i, k_, s_, p_ in zip((T, H, W), k, s, p)]
    g = torch.Generator().manual_seed(15)
    x = f16_exact(torch.randn(B, 1 + T * H * W, x_rs, generator=g))
    x[:, 0] = float("nan")                                     # cls rows must not be pooled
    x[..., Cc:] = float("nan")
    xd = x.to(_TDT[dtype]).to(_dev())
    ny = 1 + To * Ho * Wo
    y = _nan((B, ny, y_rs), dtype)
    d = L.Pool3dDesc()
    d.dtype, d.mode = _DT[dtype], L.POOL_MAX if mode == "max" else L.POOL_AVG
    d.N, d.Ti, d.Hi, d.Wi, d.C = B, T, H, W, Cc
    d.To, d.Ho, d.Wo = To, Ho, Wo
    d.kt, d.kh, d.kw, d.st, d.sh, d.sw, d.pt, d.ph, d.pw = *k, *s, *p
    d.x_row_stride, d.y_row_stride = x_rs, y_rs
    d.x_batch_stride, d.y_batch_stride = (1 + T * H * W) * x_rs, ny * y_rs
    esz = 2 if dtype == "f16" else 4
    _assert_route(_launched(lambda: L.check(lib.pv_pool3d_fwd(C.byref(d), xd.data_ptr() + x_rs * esz,
                                                              y.data_ptr() + y_rs * esz, _stream()), "pv_pool3d_fwd")),
                  ["pool3d_kernel"])
    xs = x[:, 1:, :Cc].double().reshape(B, T, H, W, Cc).permute(0, 4, 1, 2, 3)
    if mode == "max":
        ref = F.max_pool3d(xs, k, s, p)
        S = F.max_pool3d(xs.abs(), k, s, p)
    else:
        ref = F.avg_pool3d(xs, k, s, p)
        S = F.avg_pool3d(xs.abs(), k, s, p)
    got = y.cpu()
    out = got[:, 1:, :Cc].double().reshape(B, To, Ho, Wo, Cc).permute(0, 4, 1, 2, 3)
    if mode == "max":
        assert torch.equal(out, ref)                           # a max of stored values: exact
    assert_close(out, ref, S, dtype, "pool %s %s" % (mode, dtype))
    assert bool(torch.isnan(got[:, 0]).all()) and bool(torch.isnan(got[:, :, Cc:]).all())


@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("rows,groups,Cc,x_pad,y_pad", [(37, 3, 32, 8, 16), (29, 2, 96, 16, 8), (9, 2, 1024, 8, 0)])
def test_layernorm_groups_row_strides(rows, groups, Cc, x_pad, y_pad, dtype):
    """pv_layernorm with `groups` independent groups per row (per-head norms) on rows wider than groups * C."""
    lib = L.load()
    x_rs, y_rs = groups * Cc + x_pad, groups * Cc + y_pad
    g = torch.Generator().manual_seed(16 + Cc)
    x = f16_exact(torch.randn(rows, x_rs, generator=g) * 2 + 0.5)
    x[:, groups * Cc:] = float("nan")
    gamma, beta = torch.rand(Cc, generator=g) + 0.5, torch.rand(Cc, generator=g) - 0.5
    xd, gd, bd = x.to(_TDT[dtype]).to(_dev()), gamma.to(_dev()), beta.to(_dev())
    y = _nan((rows + 1, y_rs), dtype)
    kern = "layernorm_reg_kernel" if Cc <= 768 else "layernorm_kernel"
    _assert_route(_launched(lambda: L.check(lib.pv_layernorm(xd.data_ptr(), y.data_ptr(), _DT[dtype], rows, groups, Cc, x_rs, y_rs,
                                                             gd.data_ptr(), bd.data_ptr(), 1e-6, _stream()), "pv_layernorm")),
                  [kern])
    xg = x[:, :groups * Cc].double().view(rows, groups, Cc)
    mean = xg.mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(xg.var(-1, unbiased=False, keepdim=True) + 1e-6)
    ref = (xg - mean) * rstd * gamma.double() + beta.double()
    S = (xg - mean).abs() * rstd * gamma.double().abs() + beta.double().abs()
    got = y.cpu()
    assert_close(got[:rows, :groups * Cc].double().view(rows, groups, Cc), ref, S, dtype,
                 "layernorm groups %d C %d %s" % (groups, Cc, dtype))
    assert bool(torch.isnan(got[:rows, groups * Cc:]).all()) and bool(torch.isnan(got[rows:]).all())


# ---------------------------------------------------------------------------------------------------------------
# E. Squeeze-Excitation, heads, multi-view
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("N,npos,Cc,rs", [(2, 60000, 48, 56), (3, 1000, 432, 440), (1, 37, 2064, 2064)])
def test_channel_sum_large_npos(N, npos, Cc, rs, dtype):
    """fp32 atomics make the summation order arbitrary; values on a 1/8 grid keep every partial sum exact in fp32,
    so the result must equal the float64 sum BIT FOR BIT whatever the order."""
    lib = L.load()
    g = torch.Generator().manual_seed(17)
    x = torch.randint(-32, 33, (N, npos, rs), generator=g).float() / 8
    x[..., Cc:] = float("nan")
    xd = x.to(_TDT[dtype]).to(_dev())
    sums = torch.zeros(N * Cc + 8, device=_dev())
    sums[N * Cc:] = float("nan")
    _assert_route(_launched(lambda: L.check(lib.pv_channel_sum(xd.data_ptr(), _DT[dtype], rs, N, npos, Cc, sums.data_ptr(),
                                                               _stream()), "pv_channel_sum")), ["channel_sum_kernel"])
    got = sums.cpu()
    ref = x[..., :Cc].double().sum(1)
    assert torch.equal(got[:N * Cc].double().view(N, Cc), ref)
    assert bool(torch.isnan(got[N * Cc:]).all())


def test_se_gate_against_float64_mlp():
    lib = L.load()
    N, Cc, Cr, cs, npos = 3, 48, 12, 56, 1234
    g = torch.Generator().manual_seed(18)
    sums = torch.randn(N, Cc, generator=g) * npos
    w1 = torch.randn(Cr, cs, generator=g) * Cc ** -0.5
    w1[:, Cc:] = float("nan")                                  # columns past C (c_stride_w > C) are never read
    b1 = torch.randn(Cr, generator=g) * 0.1
    w2 = torch.randn(Cc, Cr, generator=g) * Cr ** -0.5 * 3
    b2 = torch.randn(Cc, generator=g) * 0.1
    dv = [t.to(_dev()).contiguous() for t in (sums, w1, b1, w2, b2)]
    gate = _nan((N * Cc + 8,), torch.float32)
    _assert_route(_launched(lambda: L.check(lib.pv_se_gate(dv[0].data_ptr(), npos, N, Cc, Cr, dv[1].data_ptr(), dv[2].data_ptr(),
                                                           dv[3].data_ptr(), dv[4].data_ptr(), cs, gate.data_ptr(), _stream()),
                                            "pv_se_gate")), ["se_gate_kernel"])
    mean = sums.double() / npos
    w1d = w1[:, :Cc].double()
    h = torch.relu(mean @ w1d.t() + b1.double())
    a = h @ w2.double().t() + b2.double()
    ref = torch.sigmoid(a)
    h_abs = mean.abs() @ w1d.abs().t() + b1.double().abs()
    S = h_abs @ w2.double().abs().t() + b2.double().abs()    # absolute terms of the gate's pre-activation
    got = gate.cpu()
    assert_close(got[:N * Cc].double().view(N, Cc), ref, S, "f32", "se gate")
    assert bool(torch.isnan(got[N * Cc:]).all())


@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("act", ["none", "relu", "swish", "gelu", "sigmoid"])
@pytest.mark.parametrize("with_gate", [True, False])
def test_scale_act_in_place(act, with_gate, dtype):
    lib = L.load()
    N, npos, Cc, rs = 2, 301, 40, 48
    g = torch.Generator().manual_seed(19)
    x = f16_exact(torch.randn(N, npos, rs, generator=g) * 3)
    x[..., Cc:] = float("nan")                                 # neighbouring channels: untouched
    gate = torch.rand(N, Cc, generator=g)
    xd, gd = x.to(_TDT[dtype]).to(_dev()), gate.to(_dev())
    _assert_route(_launched(lambda: L.check(lib.pv_scale_act(xd.data_ptr(), xd.data_ptr(), _DT[dtype], rs, rs, N, npos, Cc,
                                                             gd.data_ptr() if with_gate else None, _ACTS[act], _stream()),
                                            "pv_scale_act")), ["scale_act_kernel"])
    pre = x[..., :Cc].double() * (gate.double().unsqueeze(1) if with_gate else 1.0)
    ref = act_ref(pre, act)
    S = pre.abs()
    got = xd.cpu()
    assert_close(got[..., :Cc].double(), ref, S, dtype, "scale_act %s gate %s %s" % (act, with_gate, dtype))
    assert bool(torch.isnan(got[..., Cc:]).all())


@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("softmax", [0, 1])
@pytest.mark.parametrize("C_valid,rs", [(400, 400), (101, 112), (7, 16)])
def test_head_reduce(C_valid, rs, softmax, dtype):
    """out[n][c] = mean_p act(x[n][p][c]) for c < C_valid; the lanes past C_valid hold large garbage that must not enter
    the softmax (Kinetics-400 heads have no pad lanes, so the models never test this)."""
    lib = L.load()
    N, npos = 3, 27
    g = torch.Generator().manual_seed(20 + C_valid)
    x = f16_exact(torch.randn(N, npos, rs, generator=g) * 2)
    x[..., C_valid:] = 30.0
    xd = x.to(_TDT[dtype]).to(_dev())
    out = _nan((N * C_valid + 8,), torch.float32)
    _assert_route(_launched(lambda: L.check(lib.pv_head_reduce(xd.data_ptr(), _DT[dtype], rs, N, npos, C_valid, softmax,
                                                               out.data_ptr(), _stream()), "pv_head_reduce")),
                  ["head_reduce_kernel"])
    xv = x[..., :C_valid].double()
    if softmax:
        ref = torch.softmax(xv, -1).mean(1)
        S = ref
    else:
        ref, S = xv.mean(1), xv.abs().mean(1)
    got = out.cpu()
    assert_close(got[:N * C_valid].double().view(N, C_valid), ref, S, "f32", "head_reduce softmax %d %s" % (softmax, dtype))
    assert bool(torch.isnan(got[N * C_valid:]).all())


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_view_reduce(mode):
    lib = L.load()
    n_videos, n_views, K = 3, 30, 400
    preds = torch.randn(n_videos * n_views, K, generator=torch.Generator().manual_seed(21))
    pd = preds.to(_dev())
    out = _nan((n_videos * K + 8,), torch.float32)
    _assert_route(_launched(lambda: L.check(lib.pv_view_reduce(pd.data_ptr(), out.data_ptr(), n_videos, n_views, K, mode,
                                                               _stream()), "pv_view_reduce")), ["view_reduce"])
    v = preds.double().view(n_videos, n_views, K)
    ref = [v.sum(1), v.mean(1), v.max(1).values][mode]
    S = [v.abs().sum(1), v.abs().mean(1), v.abs().max(1).values][mode]
    got = out.cpu()
    res = got[:n_videos * K].double().view(n_videos, K)
    if mode == 2:
        assert torch.equal(res, ref)
    assert_close(res, ref, S, "f32", "view_reduce mode %d" % mode)
    assert bool(torch.isnan(got[n_videos * K:]).all())
