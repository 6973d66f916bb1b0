"""CPU: host-side logic of the engine (packing, BN folding, lowering dry-run, sharding)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from pytorchvideo_b200 import _lib as L
from pytorchvideo_b200 import parallel as PAR
from pytorchvideo_b200 import testing as TS
from pytorchvideo_b200.engine import packing as PK
from pytorchvideo_b200.engine.lower import lower_only
import pytorchvideo_b200.models.hub as PH
from pytorchvideo_b200.transforms import functional as Fv
from pytorchvideo_b200.transforms import FusedClipTransform


def test_fold_bn_matches_torch():
    torch.manual_seed(0)
    conv = nn.Conv3d(6, 10, 1, bias=True)
    bn = nn.BatchNorm3d(10).eval()
    bn.running_mean.uniform_(-1, 1); bn.running_var.uniform_(0.5, 2); bn.weight.data.uniform_(0.5, 1.5); bn.bias.data.uniform_(-1, 1)
    x = torch.randn(2, 6, 2, 3, 3)
    ref = bn(conv(x))
    s, b = PK.fold_bn(conv.bias, bn, 10, 16)
    got = F.conv3d(x, conv.weight) * s[:10].view(1, -1, 1, 1, 1) + b[:10].view(1, -1, 1, 1, 1)
    assert torch.allclose(ref, got, atol=1e-5)
    assert float(s[10:].abs().sum()) == 0 and float(b[10:].abs().sum()) == 0


def test_weight_packing_layouts():
    w = torch.randn(10, 6, 3, 1, 3)
    d = PK.pack_dense_direct(w, 8, 16, torch.float32)
    assert d.shape == (9, 8, 16)
    assert torch.equal(d[4, 2, 7], w[7, 2, 1, 0, 1]) and float(d[:, 6:, :].abs().sum()) == 0
    t = PK.pack_dense_tcgen05(w, 64, 16)
    assert t.shape == (16, 9 * 64) and t.dtype == torch.float16
    assert t[7, 4 * 64 + 2] == w[7, 2, 1, 0, 1].half() and float(t[10:].abs().sum()) == 0
    dw = PK.pack_depthwise(torch.randn(6, 1, 3, 3, 3), 8, torch.float16)
    assert dw.shape == (27, 8)


def test_tcgen05_support_predicate_is_host_only():
    lib = L.load()
    d = L.Conv3dDesc()
    d.dtype, d.N, d.Ti, d.Hi, d.Wi, d.Ci = L.PV_F16, 2, 8, 14, 14, 256
    d.To, d.Ho, d.Wo, d.Co = 8, 14, 14, 256
    d.kt, d.kh, d.kw, d.st, d.sh, d.sw, d.pt, d.ph, d.pw, d.dt, d.dh, d.dw = 1, 3, 3, 1, 1, 1, 0, 1, 1, 1, 1, 1
    d.groups, d.x_row_stride, d.y_row_stride, d.ci_pad64 = 1, 256, 256, 256
    assert lib.pv_conv3d_tcgen05_supported(C.byref(d)) == 1
    d.dtype = L.PV_F32
    assert lib.pv_conv3d_tcgen05_supported(C.byref(d)) == 0
    d.dtype, d.x_row_stride = L.PV_F16, 260
    assert lib.pv_conv3d_tcgen05_supported(C.byref(d)) == 0


def _desc(ci, co, k, pad, ci_pad64, T=8, H=14, W=14, xrs=None):
    d = L.Conv3dDesc()
    d.dtype, d.N, d.Ti, d.Hi, d.Wi, d.Ci = L.PV_F16, 2, T, H, W, ci
    d.kt, d.kh, d.kw = k
    d.pt, d.ph, d.pw = pad
    d.st = d.sh = d.sw = d.dt = d.dh = d.dw = 1
    d.To, d.Ho, d.Wo, d.Co = T + 2 * pad[0] - k[0] + 1, H + 2 * pad[1] - k[1] + 1, W + 2 * pad[2] - k[2] + 1, co
    d.groups, d.x_row_stride, d.y_row_stride, d.ci_pad64 = 1, xrs or ci, co, ci_pad64
    return d


def test_narrow_input_dispatch_is_decided_on_the_host():
    """C_in < 64 with the weights packed at the un-padded per-tap extent: 16 / 32 go to the narrow TMA mode,
    the other widths to the gather-fed kernel; both predicates are pure host code (no GPU here)."""
    lib = L.load()
    for ci, k, pad in [(32, (3, 1, 1), (1, 0, 0)), (16, (1, 3, 3), (0, 1, 1)), (8, (1, 3, 3), (0, 1, 1)),
                       (24, (1, 1, 1), (0, 0, 0)), (56, (1, 1, 1), (0, 0, 0)), (4, (1, 7, 7), (0, 3, 3))]:
        assert lib.pv_conv3d_tcgen05_supported(C.byref(_desc(ci, 16, k, pad, ci))) == 1, (ci, k)
    # 5x7x7 over 8 channels: 245 taps > 64 validity bits of the gather kernel and not a narrow-TMA width
    assert lib.pv_conv3d_tcgen05_supported(C.byref(_desc(8, 16, (5, 7, 7), (2, 3, 3), 8))) == 0
    # a channel slice whose row stride is not a multiple of 16 bytes cannot be a TMA / 16-byte cp.async source
    assert lib.pv_conv3d_tcgen05_supported(C.byref(_desc(32, 16, (1, 1, 1), (0, 0, 0), 32, xrs=36))) == 0
    # 12 channels is neither 4 nor a multiple of 8
    assert lib.pv_conv3d_tcgen05_supported(C.byref(_desc(12, 16, (1, 1, 1), (0, 0, 0), 12))) == 0


def test_lowering_slowfast_dry_run():
    m = PH.slowfast_r50().eval()
    clip = torch.zeros(2, 3, 32, 224, 224)
    plan, out_shape = lower_only(m, TS.slowfast_inputs(clip))
    assert out_shape == (2, 400)
    names = [n for n, _ in plan.ops]
    # 2 stems (conv+pool each), 4 fusion convs, (3+4+6+3)*2 blocks * 3 convs + 8 shortcuts, head; the 13 blocks of the
    # Fast pathway's res2-res3 (3 convs each + their 2 projection shortcuts) are ONE fused launch each
    n_conv = plan.stats["tcgen05"] + plan.stats["direct"]
    assert plan.stats["fused_block"] == 7
    assert n_conv == 2 + 4 + 2 * (16 * 3 + 4) + 1 - (7 * 3 + 2)
    assert plan.stats["tcgen05"] == n_conv        # every C_in%8==0 dense conv goes to the tensor cores
    assert any(n.endswith("multipathway_fusion.conv_fast_to_slow") for n in names)
    assert "blocks.6.output_pool" in names


@pytest.mark.parametrize("case", sorted(TS.MODEL_CASES))
def test_every_model_case_lowers_on_the_host(case):
    """Host-side dry run (no GPU): every hub entry that has a golden lowers to a static plan with the right
    output shape, no CUDA-core dense convolution left in f16 mode except a 3-channel stem the window mode
    cannot take, and a depthwise op for every depthwise conv of the tree."""
    hub, kw, B, T, H, W, is_sf = TS.MODEL_CASES[case]
    m = getattr(PH, hub)(**kw).eval()
    clip = torch.zeros(B, 3, T, H, W)
    plan, out_shape = lower_only(m, TS.slowfast_inputs(clip) if is_sf else clip)
    assert out_shape == (B, 400)
    n_dw = sum(1 for mod in m.modules() if isinstance(mod, torch.nn.Conv3d) and mod.groups > 1)
    if "mvit" not in case:          # MViT shares one pooling conv across heads: counted per use, not per module
        assert plan.stats["depthwise"] == n_dw
    assert plan.stats["direct"] <= 1
    assert plan.stats["tcgen05"] > 0


def test_lowering_f32_mode_uses_no_tensor_core_path():
    m = PH.x3d_xs().eval()
    plan, out_shape = lower_only(m, torch.zeros(1, 3, 4, 160, 160), dtype="f32")
    assert out_shape == (1, 400) and plan.stats["tcgen05"] == 0 and plan.stats["depthwise"] == 27


def test_wrong_channel_count_raises_runtimeerror():
    # reference behaviour asserted by tests/test_models_x3d.py:64-67 and test_models_slowfast.py:119-122
    m = PH.x3d_xs().eval()
    with pytest.raises(RuntimeError):
        lower_only(m, torch.zeros(1, 4, 4, 160, 160))


def test_concat_is_fused_into_channel_slices():
    m = PH.slowfast_r50().eval()
    plan, _ = lower_only(m, TS.slowfast_inputs(torch.zeros(1, 3, 32, 224, 224)))
    # after stage 0 the slow tensor (64 ch) and the fused lateral (16 ch) share an 80-wide buffer
    from pytorchvideo_b200.engine.plan import TRef
    assert not any(n.startswith("cat") for n, _ in plan.ops)


def test_transform_plan_matches_reference_formulas():
    tr = FusedClipTransform(16, (0.45,) * 3, (0.225,) * 3, short_side=256, crop=("center", 224))
    idx, hw, win, flip = tr.plan((3, 64, 1080, 1920))
    assert flip is False
    assert idx.tolist() == [0, 4, 8, 12, 16, 21, 25, 29, 33, 37, 42, 46, 50, 54, 58, 63]
    assert hw == (256, 455) and win == (16, 116, 224, 224)
    # host tables are the oracle's
    from oracle import transforms_ref as O
    for a, b in zip(Fv.bilinear_table(1920, 455), O.bilinear_table(1920, 455)):
        assert np.array_equal(a, b)
    assert Fv.uniform_crop_window(20, 40, 16, 2) == O.uniform_crop_window(20, 40, 16, 2)


def test_shard_bounds_cover_batch_exactly():
    for n in (0, 1, 7, 8, 64, 257):
        for w in (1, 2, 3, 8):
            spans = [PAR.shard_bounds(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_lowering_mvit_dry_run_counts_match_the_reference_macs():
    m = PH.mvit_base_16x4().eval()
    plan, out_shape = lower_only(m, torch.zeros(1, 3, 16, 224, 224))
    assert out_shape == (1, 400)
    gmac = sum(x["flops"] for x in plan.meta) / 2e9
    assert abs(gmac - 70.60) < 0.05            # SURVEY section 6: 70.60 GMAC/clip hook-counted on the reference
    assert plan.stats["attention"] == 16 and plan.stats["tcgen05"] == 1 + 16 * 4 + 3 + 1


def test_slowfast_pathways_are_scheduled_on_two_lanes():
    """engine/plan.py lanes: the Slow and Fast pathways are independent until each lateral fusion, so they
    are enqueued on two CUDA streams (graph branches).  The only cross-lane edges are read-after-write: the
    first Slow op of stage k+1 waits for the lateral conv of stage k, and the head waits for the Fast pool."""
    m = PH.slowfast_r50().eval()
    plan, _ = lower_only(m, TS.slowfast_inputs(torch.zeros(1, 3, 32, 224, 224)))
    plan._schedule()
    sc = plan.sched
    assert sc["lanes"] == [0, 1]
    names = [n for n, _ in plan.ops]
    lane = dict(zip(names, plan.op_lane))
    assert lane["blocks.1.multipathway_blocks.0.res_blocks.0.branch2.conv_a"] == 0
    assert lane["blocks.1.multipathway_blocks.1.res_blocks.0.fused"] == 1     # Fast-pathway blocks: one fused launch each
    assert lane["blocks.1.multipathway_fusion.conv_fast_to_slow"] == 1
    edges = [(names[j], names[i]) for i, w in enumerate(sc["waits"]) for j in w]
    for k in range(4):
        assert ("blocks.%d.multipathway_fusion.conv_fast_to_slow" % k,
                "blocks.%d.multipathway_blocks.0.res_blocks.0.branch1" % (k + 1)) in edges
    assert ("blocks.5.pool.1", "blocks.6.proj") in edges
    assert len(edges) == 5                       # nothing else crosses lanes
    # every op that is waited for records an event
    assert sc["signals"] == {names.index(a) for a, _ in edges}
    assert plan.stats["fused_block"] == 7 and len(names) == 103               # res2 + res3 of the Fast pathway (3 + 4 blocks)
    # single-lane models keep one stream
    p2, _ = lower_only(PH.slow_r50().eval(), torch.zeros(1, 3, 8, 224, 224))
    p2._schedule()
    assert p2.sched["lanes"] == [0] and not any(p2.sched["waits"])


@pytest.mark.parametrize("name", TS.LAYER_CASES)
def test_layer_modules_lower_on_the_host(name):
    """Every `pytorchvideo.layers` / stem / head module has a lowering (no ``NotImplementedError`` forward)."""
    g = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "layers.pt"), weights_only=False)[name]
    m, x, thw = TS.build_layer_case(name)
    plan, shape = lower_only(m, torch.zeros(x.shape), extra=() if thw is None else (tuple(thw),))
    assert tuple(shape) == tuple(g["output"].shape)
    assert (plan.aux if thw is not None else None) == g["thw_out"]


def test_lowering_accepts_the_reference_modules_themselves():
    """INTEGRATION.md route 2: the lowering dispatches on the reference's class / attribute NAMES, so the reference's
    own model objects lower to the same plan as this package's trees.  tests/golden/lowering.pt holds the reference
    models' module trees and the plans lowered from them (oracle/gen_golden.py)."""
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lowering.pt"), weights_only=False)
    assert sorted(gold) == ["mvit_base_16x4", "slowfast_r50", "x3d_xs"]
    for name, g in gold.items():
        mine = getattr(PH, name)().eval()
        assert [(n, type(m).__name__) for n, m in mine.named_modules()] == g["modules"]
        shapes = g["input_shapes"]
        inp = [torch.zeros(s) for s in shapes] if len(shapes) > 1 else torch.zeros(shapes[0])
        p_mine, s_mine = lower_only(mine, inp)
        assert tuple(s_mine) == g["output_shape"]
        assert [n for n, _ in p_mine.ops] == g["ops"]
        assert p_mine.stats == g["stats"]


def test_modules_deepcopy_without_their_compiled_plans():
    """The reference's transmuter deep-copies models (accelerator/deployment/common/model_transmuter.py); compiled plans
    (device buffers, graphs, ctypes descriptors) are derived data and must not travel with a copy or a pickle."""
    import copy
    import ctypes
    m = PH.x3d_xs().eval()
    m.__dict__["_pv_cache"] = {"k": ctypes.pointer(ctypes.c_int(1))}
    m.blocks[1].__dict__["_pv_cache"] = {"k": ctypes.pointer(ctypes.c_int(1))}
    m2 = copy.deepcopy(m)
    assert "_pv_cache" not in m2.__dict__ and "_pv_cache" not in m2.blocks[1].__dict__
    assert "_pv_cache" in m.__dict__
    assert list(m2.state_dict()) == list(m.state_dict())


@pytest.mark.parametrize("case", sorted(TS.DETECTION_CASES))
def test_detection_models_lower_on_the_host(case):
    """DetectionBBoxNetwork (trunk + RoIAlign head, models/net.py:47-74, head.py:394-482): one plan whose last ops are
    roi_align -> spatial max pool -> proj; the [K, 5] boxes are a raw fp32 plan input."""
    from pytorchvideo_b200.engine.lower import lower_only
    model, inp, boxes, is_sf = TS.build_detection_case(case, PH)
    ins = (list(inp) if is_sf else [inp]) + [boxes]
    plan, shape = lower_only(model, ins)
    K = boxes.shape[0]
    assert tuple(shape)[:2] == (K, 80)
    names = [n for n, _ in plan.ops]
    assert any(n.endswith("roi_layer") for n in names) and any(n.endswith("pool_spatial") for n in names)
    # dilated res5 (conv_b dilation (1,2,2), spatial stride 1) keeps the 1/16 feature map the head's spatial_scale assumes
    assert sum(1 for n in names if n.endswith("roi_layer")) == 1
    with pytest.raises(RuntimeError):
        lower_only(model, (list(inp) if is_sf else [inp]) + [torch.zeros(3, 6)])        # RoIAlignRotated boxes
    with pytest.raises(RuntimeError):
        lower_only(model, (list(inp) if is_sf else [inp]) + [torch.zeros(0, 5)])


def test_detection_state_dict_and_repr_follow_the_reference():
    m = PH.slowfast_r50_detection()
    sd = m.state_dict()
    assert "model.blocks.0.multipathway_blocks.0.conv.weight" in sd and "detection_head.proj.weight" in sd
    assert sd["detection_head.proj.weight"].shape == (80, 2304)
    assert repr(m.detection_head.roi_layer) == "RoIAlign(output_size=(7, 7), spatial_scale=0.0625, sampling_ratio=0, aligned=False)"
    s = PH.slow_r50_detection()
    assert s.state_dict()["detection_head.proj.weight"].shape == (80, 2048)
    assert type(s.detection_head.pool).__name__ == "AvgPool3d" and tuple(s.detection_head.pool.kernel_size) == (4, 1, 1)


def test_mvit_fp32_trunk_and_fused_pooling_plan():
    """f16 engine, MViT-B: the residual stream is fp32 (every residual add is a pv_add_layernorm launch fused with the
    LayerNorm that follows - norm2 / next block's norm1 / norm_embed), pooled K and V share one depthwise + one
    LayerNorm launch, no cls copy launches except on the norm-less skip path; f32 parity mode keeps the plain lowering."""
    from pytorchvideo_b200 import _lib as L
    m = PH.mvit_base_16x4(spatial_size=112, temporal_size=8).eval()
    x = torch.zeros(2, 3, 8, 112, 112)
    plan = lower_only(m, x)[0]
    names = [mm["name"] for mm in plan.meta]
    assert plan.trunk32 and len(names) == 165
    assert names.count("blocks.0.norm1") == 1 and not any(n.endswith(".norm1") for n in names if not n.startswith("blocks.0."))
    assert sum(n.endswith(".norm2") for n in names) == 16 and sum(n.endswith(".add") for n in names) == 16
    assert sum(n.endswith(".pool_kv.dwconv") for n in names) == 16 and not any(".pool_k." in n or ".pool_v." in n for n in names)
    assert [n for n in names if n.endswith(".cls")] == ["blocks.%d.pool_skip.cls" % i for i in (1, 3, 14)]
    assert "norm_embed" not in names                       # fused into blocks.15.add
    # the trunk tensors are f32 buffers, everything a GEMM reads is f16
    dts = {b.dt for b in plan.bufs}
    assert dts == {L.PV_F16, L.PV_F32}
    plan32 = lower_only(m, x, dtype="f32")[0]
    n32 = [mm["name"] for mm in plan32.meta]
    assert not plan32.trunk32 and "norm_embed" in n32 and not any(n.endswith(".add") for n in n32)


def test_numa_helpers_are_safe_without_sysfs(tmp_path):
    from pytorchvideo_b200 import parallel as PAR
    assert PAR._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert PAR._parse_cpulist("") == set()
    # no GPU / no sysfs entry: a silent no-op, never an exception (bench.py calls it on every multi-rank run)
    assert PAR.gpu_numa_cpus(0, sysfs=str(tmp_path)) == (None, None)
    assert PAR.bind_to_gpu_numa(0) is None


@pytest.mark.parametrize("variant", ["default", "no_cls", "no_sep_pos", "pool_max", "separate_qkv", "dim_mul_in_att",
                                     "residual_pool_off", "no_kv_pool"])
def test_mvit_variants_lower_on_the_host(variant):
    """create_multiscale_vision_transformers options (models/vision_transformers.py:185-437) all reach a plan in both
    precision modes: fused K|V pooling where the two branches are depthwise convs with LayerNorms, separate launches
    otherwise; the fp32 trunk only in the f16 engine."""
    from pytorchvideo_b200.models.vision_transformers import create_multiscale_vision_transformers as mk
    base = dict(spatial_size=64, temporal_size=4, depth=4, embed_dim_mul=[[1, 2.0], [3, 2.0]], atten_head_mul=[[1, 2.0], [3, 2.0]],
                pool_q_stride_size=[[1, 1, 2, 2], [3, 1, 2, 2]], pool_kv_stride_adaptive=[1, 4, 4], pool_kvq_kernel=[3, 3, 3])
    kw = {"default": {}, "no_cls": {"cls_embed_on": False}, "no_sep_pos": {"sep_pos_embed": False},
          "pool_max": {"pool_kv_stride_adaptive": None, "pool_kv_stride_size": [[0, 1, 2, 2]], "pooling_mode": "max"},
          "separate_qkv": {"separate_qkv": True}, "dim_mul_in_att": {"dim_mul_in_att": True},
          "residual_pool_off": {"residual_pool": False},
          "no_kv_pool": {"pool_kv_stride_adaptive": None, "pool_q_stride_size": None}}[variant]
    m = mk(**{**base, **kw}).eval()
    x = torch.zeros(1, 3, 4, 64, 64)
    for dt in ("f16", "f32"):
        plan, shp = lower_only(m, x, dtype=dt)
        assert shp == (1, 400)
        names = [mm["name"] for mm in plan.meta]
        assert plan.trunk32 == (dt == "f16")
        assert sum(n.endswith(".attn.core") for n in names) == 4
        if variant in ("default", "separate_qkv"):
            assert sum(n.endswith(".pool_kv.dwconv") for n in names) == 4 and not any(".pool_k." in n for n in names)
        if variant == "no_kv_pool":
            assert not any(".pool_" in n and ".attn." in n for n in names)


@pytest.mark.parametrize("stem,k,s,p,W,mutation", [
    ("x3d_l", (1, 3, 3), (1, 2, 2), (0, 1, 1), 312, "second W tile one pixel early"),
    ("slow", (1, 7, 7), (1, 2, 2), (0, 3, 3), 224, "corner tap zeroed"),
    ("i3d", (5, 7, 7), (1, 2, 2), (2, 3, 3), 224, "last temporal tap zeroed"),
])
def test_entry_point_tolerance_detects_one_missing_tap(stem, k, s, p, W, mutation):
    """The per-element bound of tests/test_gpu_entry_points.py accepts one f16 rounding of the float64 reference but
    rejects the reference of a convolution with one tap missing, or with its second 128-pixel W tile shifted."""
    from test_gpu_entry_points import conv_reference, worst_ratio
    g = torch.Generator().manual_seed(len(stem))
    T = 3 if k[0] > 1 else 1
    x = TS.f16_exact(torch.randn(2, 3, T, 16, W, generator=g))
    w = TS.f16_exact(torch.randn(24, 3, *k, generator=g) * (2.0 / (3 * k[0] * k[1] * k[2])) ** 0.5)
    scale, bias = torch.rand(24, generator=g) + 0.5, torch.rand(24, generator=g) - 0.5
    ref, S = conv_reference(x, w, scale, bias, s, p, act="relu")
    assert worst_ratio(TS.f16_exact(ref.float()), ref, S, "f16") <= 1.0
    assert worst_ratio(ref.float(), ref, S, "f32") <= 1.0
    if mutation.startswith("second W tile"):
        assert ref.shape[-1] == 156
        bad = ref.clone()
        bad[..., 128:] = ref[..., 127:-1]
    else:
        w2 = w.clone()
        if mutation == "corner tap zeroed":
            w2[:, :, 0, -1, -1] = 0
        else:
            w2[:, :, -1] = 0
        bad, _ = conv_reference(x, w2, scale, bias, s, p, act="relu")
    for dt in ("f16", "f32"):
        assert worst_ratio(bad, ref, S, dt) > 4.0, (mutation, dt)
