"""Golden-vector generator (runs ONLY in the authoring container, where /root/reference exists).

Imports the unmodified reference (with the 3-symbol fvcore shim in oracle/shim), loads this
repo's deterministic weights into the reference models with ``load_state_dict(strict=True)``
(this also proves state_dict / module-tree compatibility), runs the reference CPU forward and
stores the outputs as small fixtures under tests/golden/.  It also pins the oracle: the
interpreter in oracle/interp.py, run over the REAL reference modules, must reproduce the
reference output bit-for-bit, and the numpy transform restatement must match the reference's
own transforms.

    PYTHONPATH=oracle/shim:/root/reference python oracle/gen_golden.py [--only name]
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "shim"))
sys.path.insert(1, "/root/reference")

GOLD = os.path.join(ROOT, "tests", "golden")


def gen_models(only=None):
    import pytorchvideo.models.hub as RH            # the reference
    import pytorchvideo_b200.models.hub as PH       # this repo's parameter containers
    from pytorchvideo_b200 import testing as TS
    from oracle.interp import oracle_forward
    for case, (hub, kw, B, T, H, W, is_sf) in TS.MODEL_CASES.items():
        if only and case != only:
            continue
        t0 = time.time()
        grid = TS.CASE_OPTS.get(case, {}).get("f16_grid", False)
        mine = getattr(PH, hub)(**kw)
        TS.randomize_model(mine, seed=1234, f16_weights=grid)
        ref = getattr(RH, hub)(pretrained=False, **kw)
        ref.load_state_dict(mine.state_dict(), strict=True)
        ref.eval()
        clip = TS.synthetic_clip(B, T, H, W, seed=42, f16_values=grid)
        with torch.no_grad():
            inp = TS.slowfast_inputs(clip) if is_sf else clip
            out_ref = ref(list(inp) if is_sf else inp)          # list() - the reference mutates it
            inp = TS.slowfast_inputs(clip) if is_sf else clip
            out_orc_on_mine = oracle_forward(mine, inp)
            # (the big-batch cases pin the oracle on the product tree only: one oracle pass instead of two)
            out_orc_on_ref = oracle_forward(ref, inp) if B * T * H * W <= 4 * 32 * 224 * 224 else out_orc_on_mine
        assert torch.equal(out_ref, out_orc_on_ref), "oracle != reference on reference modules (%s)" % case
        assert torch.equal(out_ref, out_orc_on_mine), "oracle != reference on product tree (%s)" % case
        torch.save({"case": case, "hub": hub, "batch": B, "T": T, "H": H, "W": W, "weight_seed": 1234,
                    "input_seed": 42, "f16_grid": grid, "output": out_ref.clone(),
                    "input_checksum": TS.tensor_checksum(clip),
                    "state_checksum": TS.state_checksum(mine)},
                   os.path.join(GOLD, "model_%s.pt" % case))
        print("%-14s ok  out %s  |out|max %.4f  (%.1fs)" % (case, tuple(out_ref.shape), float(out_ref.abs().max()),
                                                            time.time() - t0), flush=True)


def gen_transforms():
    import pytorchvideo.transforms.functional as RF   # reference functional (imports fine without av)
    from pytorchvideo.transforms import transforms as RT
    import torchvision.transforms as TV
    from oracle import transforms_ref as O
    from pytorchvideo_b200 import testing as TS
    out = {}
    # (1) temporal indices: oracle restatement vs reference on a grid + the reference's known answer
    grid = {}
    for t in list(range(1, 80)) + [100, 128, 250, 300]:
        for n in list(range(1, 40)) + [64, 100, 128]:
            x = torch.arange(t).view(1, t, 1, 1)
            ref_idx = RF.uniform_temporal_subsample(x, n).view(-1).numpy()
            assert np.array_equal(ref_idx, O.linspace_indices(t, n)), (t, n)
            if (t, n) in ((20, 10), (64, 16), (64, 32), (32, 8), (300, 128), (7, 13)):
                grid["%d_%d" % (t, n)] = ref_idx.astype(np.int64)
    out["indices"] = grid
    # (2) small-clip chain goldens (reference order: subsample, /255, normalize, scale, center crop)
    cases = []
    for (T, H, W, n, side, crop, seed) in [(20, 40, 60, 10, 24, 16, 1), (9, 61, 37, 4, 30, 28, 2),
                                           (16, 48, 48, 16, 48, 32, 3), (12, 90, 160, 5, 32, 32, 4)]:
        clip = TS.synthetic_u8_clip(T, H, W, seed=seed)
        mean, std = (0.45, 0.45, 0.45), (0.225, 0.225, 0.225)
        chain = TV.Compose([RT.UniformTemporalSubsample(n), RT.Div255(), RT.Normalize(mean, std),
                            RT.ShortSideScale(side), TV.CenterCrop(crop)])
        ref = chain(clip)
        orc = O.val_chain(clip.numpy(), n, mean, std, side, crop)
        err = float(np.abs(ref.numpy() - orc).max())
        assert err <= 2e-6, ("oracle transform chain deviates from the reference", err)
        cases.append({"T": T, "H": H, "W": W, "n": n, "side": side, "crop": crop, "seed": seed,
                      "mean": mean, "std": std, "out": ref.clone(), "oracle_max_err": err})
    out["chain_small"] = cases
    # (3) BASELINE config 5 at full size: keep a strided sample + checksums
    clip = TS.synthetic_u8_clip(64, 1080, 1920, seed=0)
    mean, std = (0.45, 0.45, 0.45), (0.225, 0.225, 0.225)
    chain = TV.Compose([RT.UniformTemporalSubsample(16), RT.Div255(), RT.Normalize(mean, std),
                        RT.ShortSideScale(256), TV.CenterCrop(224)])
    t0 = time.time()
    ref = chain(clip)
    dt = time.time() - t0
    orc = O.val_chain(clip.numpy(), 16, mean, std, 256, 224)
    err = float(np.abs(ref.numpy() - orc).max())
    assert err <= 2e-6, err
    out["chain_full"] = {"T": 64, "H": 1080, "W": 1920, "n": 16, "side": 256, "crop": 224, "seed": 0,
                         "mean": mean, "std": std, "sample": ref[:, ::5, ::7, ::9].clone(),
                         "checksum": TS.tensor_checksum(ref), "ref_seconds": dt, "oracle_max_err": err}
    # (4) bilinear tables: oracle vs ATen-extracted weights
    import torch.nn.functional as F
    for (i, o) in [(1080, 256), (1920, 455), (320, 224), (7, 13), (224, 224), (61, 30), (240, 320)]:
        eye = torch.eye(i).view(1, i, 1, i)
        w = F.interpolate(eye, size=(1, o), mode="bilinear", align_corners=False)[0, :, 0, :].numpy()
        i0, i1, l1 = O.bilinear_table(i, o)
        W = np.zeros((i, o), np.float32)
        for j in range(o):
            W[i0[j], j] += np.float32(1) - l1[j]
            W[i1[j], j] += l1[j]
        assert np.array_equal(W, w), ("bilinear table mismatch", i, o)
    # (5) crops (reference known answers: tests/test_transforms.py:199-226, 334-346)
    out["uniform_crop"] = {}
    for (h, w, size) in [(20, 40, 16), (40, 20, 16), (30, 30, 10)]:
        for idx in range(3):
            x = torch.arange(h * w, dtype=torch.float32).view(1, 1, h, w)
            ref = RF.uniform_crop(x, size, idx)
            y, xo, hh, ww = O.uniform_crop_window(h, w, size, idx)
            assert torch.equal(ref, x[:, :, y:y + hh, xo:xo + ww])
            out["uniform_crop"]["%d_%d_%d_%d" % (h, w, size, idx)] = (y, xo)
    # (6) default TRAIN chain of the reference factory under a fixed seed (global torch RNG): pins the order
    #     and arithmetic of the random draws (RandomShortSideScale, torchvision RandomCrop / RandomHorizontalFlip)
    from pytorchvideo.transforms import create_video_transform as ref_factory
    tr_cases = []
    for (T, H, W, n, lo, hi, crop, seed) in [(20, 40, 60, 10, 24, 32, 16, 11), (9, 61, 37, 4, 30, 40, 28, 12),
                                             (12, 90, 160, 5, 32, 48, 32, 13), (16, 48, 48, 16, 32, 32, 32, 14),
                                             (10, 36, 36, 6, 20, 28, 20, 15), (8, 30, 50, 8, 16, 24, 16, 16)]:
        clip = TS.synthetic_u8_clip(T, H, W, seed=seed)
        chain = ref_factory(mode="train", num_samples=n, min_size=lo, max_size=hi, crop_size=crop)
        torch.manual_seed(1000 + seed)
        ref = chain(clip)
        # the same draws, made by hand in the order the Compose makes them
        torch.manual_seed(1000 + seed)
        side = int(torch.randint(lo, hi + 1, (1,)).item())
        nh, nw = O.short_side_size(H, W, side)
        if (nh, nw) == (crop, crop):
            i = j = 0
        else:
            i = int(torch.randint(0, nh - crop + 1, size=(1,)).item())
            j = int(torch.randint(0, nw - crop + 1, size=(1,)).item())
        flip = bool(torch.rand(1) < 0.5)
        orc = O.train_chain(clip.numpy(), n, (0.45,) * 3, (0.225,) * 3, side, crop, i, j, flip)
        err = float(np.abs(ref.numpy() - orc).max())
        assert err <= 2e-6, ("oracle train chain deviates from the reference", err)
        tr_cases.append({"T": T, "H": H, "W": W, "n": n, "min_size": lo, "max_size": hi, "crop": crop, "seed": seed,
                         "rng_seed": 1000 + seed, "draws": (side, i, j, flip), "out": ref.clone(), "oracle_max_err": err})
    assert any(c["draws"][3] for c in tr_cases) and not all(c["draws"][3] for c in tr_cases), "want flipped and unflipped cases"
    out["train_small"] = tr_cases
    # (7) SlowFast pathway packing (pytorchvideo_trainer/datamodule/transforms.py:99-138 restated: the trainer
    #     package is not importable without hydra/lightning): slow = index_select(frames, 1, linspace(0, T-1, T//alpha).long())
    out["pack_pathway"] = {"%d_%d" % (t, a): torch.linspace(0, t - 1, t // a).long() for (t, a) in [(32, 4), (64, 4), (16, 4), (32, 8), (8, 4)]}
    torch.save(out, os.path.join(GOLD, "transforms.pt"))
    print("transforms ok (full-size reference chain took %.2fs)" % dt, flush=True)


def gen_layers():
    """Layer-level goldens from the REAL reference classes (same constructor arguments, weights copied with
    load_state_dict(strict=True)): ConvReduce3D, Conv2plus1d (both orders), Mlp, MultiScaleAttention,
    MultiScaleBlock, positional encoding, PatchEmbed, ViT head.  Also pins the oracle on each of them."""
    import pytorchvideo.layers as RL
    import pytorchvideo.layers.convolutions as RC
    import pytorchvideo.models.head as RHd
    import pytorchvideo.models.stem as RSt
    from functools import partial
    import torch.nn as nn
    from pytorchvideo_b200 import testing as TS
    from oracle.interp import oracle_forward
    ln = partial(nn.LayerNorm, eps=1e-6)
    ref_make = {
        "conv_reduce_sum": lambda: RC.ConvReduce3D(in_channels=16, out_channels=32, kernel_size=((1, 1, 1), (3, 3, 3), (1, 3, 3)),
                                                   stride=((1, 1, 1), (1, 1, 1), None), padding=((0, 0, 0), (1, 1, 1), (0, 1, 1)),
                                                   bias=(False, True, None), reduction_method="sum"),
        "conv_reduce_cat": lambda: RC.ConvReduce3D(in_channels=16, out_channels=24, kernel_size=((1, 1, 1), (3, 1, 1)),
                                                   padding=((0, 0, 0), (1, 0, 0)), reduction_method="cat"),
        "conv2plus1d_xy_first": lambda: RC.create_conv_2plus1d(in_channels=16, out_channels=32, inner_channels=24,
                                                               conv_xy_first=True, stride=(1, 2, 2)),
        "conv2plus1d": lambda: RC.create_conv_2plus1d(in_channels=16, out_channels=32, stride=(2, 1, 1)),
        "mlp": lambda: RL.Mlp(in_features=96, hidden_features=384, out_features=192),
        "attention_pool_qkv": lambda: RL.MultiScaleAttention(192, num_heads=2, qkv_bias=True, kernel_q=(3, 3, 3), kernel_kv=(3, 3, 3),
                                                             stride_q=(1, 2, 2), stride_kv=(1, 4, 4), norm_layer=ln, residual_pool=False),
        "attention_residual_pool_nocls": lambda: RL.MultiScaleAttention(64, num_heads=2, kernel_kv=(3, 3, 3), stride_kv=(1, 2, 2),
                                                                        has_cls_embed=False, norm_layer=ln, residual_pool=True),
        "block_widen_pool": lambda: RL.MultiScaleBlock(96, 192, 1, qkv_bias=True, norm_layer=ln, attn_norm_layer=ln,
                                                       kernel_q=(3, 3, 3), kernel_kv=(3, 3, 3), stride_q=(1, 2, 2), stride_kv=(1, 2, 2)),
        "block_dim_mul_in_att": lambda: RL.MultiScaleBlock(64, 128, 2, qkv_bias=True, norm_layer=ln, attn_norm_layer=ln,
                                                           dim_mul_in_att=True, kernel_kv=(3, 3, 3), stride_kv=(1, 2, 2)),
        "posenc": lambda: RL.SpatioTemporalClsPositionalEncoding(96, (4, 7, 7), sep_pos_embed=True, has_cls=True),
        "patch_embed": lambda: RSt.create_conv_patch_embed(in_channels=3, out_channels=96, conv_kernel_size=(3, 7, 7),
                                                           conv_stride=(2, 4, 4), conv_padding=(1, 3, 3)),
        "vit_head": lambda: RHd.create_vit_basic_head(in_features=192, out_features=40, seq_pool_type="cls"),
    }
    out = {}
    for name in TS.LAYER_CASES:
        mine, x, thw = TS.build_layer_case(name)
        ref = ref_make[name]()
        ref.load_state_dict(mine.state_dict(), strict=True)
        ref.eval()
        with torch.no_grad():
            if thw is None:
                y_ref, thw_ref = ref(x), None
                y_orc, thw_orc = oracle_forward(mine, x), None
            else:
                y_ref, thw_ref = ref(x, list(thw))
                y_orc, thw_orc = oracle_forward(mine, x, thw)
        assert torch.equal(y_ref, y_orc), "oracle != reference on layer case %s" % name
        assert thw_ref is None or list(thw_ref) == list(thw_orc)
        out[name] = {"output": y_ref.clone(), "thw_out": None if thw_ref is None else list(thw_ref),
                     "state_checksum": TS.state_checksum(mine), "input_checksum": TS.tensor_checksum(x)}
        print("layer %-30s ok  out %s  thw %s" % (name, tuple(y_ref.shape), out[name]["thw_out"]), flush=True)
    torch.save(out, os.path.join(GOLD, "layers.pt"))


def gen_detection():
    """Detection goldens (SURVEY 8 row f3): the reference's slow_r50_detection / slowfast_r50_detection (trunk +
    ResNetRoIHead with torchvision.ops.RoIAlign) on small clips, and torchvision.ops.roi_align itself on an op-level
    case.  Pins oracle/interp.py (roi_align_ref, f_ResNetRoIHead, f_DetectionBBoxNetwork) bit-for-bit."""
    import torchvision
    import pytorchvideo.models.hub as RH
    import pytorchvideo_b200.models.hub as PH
    from pytorchvideo_b200 import testing as TS
    from oracle.interp import oracle_forward, roi_align_ref
    out = {"torchvision": torchvision.__version__}
    x, boxes, settings = TS.roi_align_case()
    ra = []
    for osz, scale, sr in settings:
        ref = torchvision.ops.roi_align(x, boxes, osz, scale, sr, False)
        assert torch.equal(ref, roi_align_ref(x, boxes, osz, scale, sr)), "roi_align_ref != torchvision (%s)" % (osz,)
        ra.append(ref.clone())
    out["roi_align"] = {"outputs": ra, "input_checksum": TS.tensor_checksum(x), "boxes": boxes.clone()}
    print("roi_align op case ok (%d settings)" % len(settings), flush=True)
    for case, (hub, kw, B, T, H, W, is_sf, K) in TS.DETECTION_CASES.items():
        t0 = time.time()
        mine, inp, bx, _ = TS.build_detection_case(case, PH)
        ref = getattr(RH, hub)(pretrained=False, **kw)
        ref.load_state_dict(mine.state_dict(), strict=True)
        ref.eval()
        assert repr(ref.detection_head.roi_layer) == repr(mine.detection_head.roi_layer)
        with torch.no_grad():
            y_ref = ref(list(inp) if is_sf else inp, bx)
            y_orc_ref = oracle_forward(ref, list(inp) if is_sf else inp, bx)
            y_orc_mine = oracle_forward(mine, list(inp) if is_sf else inp, bx)
        assert torch.equal(y_ref, y_orc_ref), "oracle != reference on reference modules (%s)" % case
        assert torch.equal(y_ref, y_orc_mine), "oracle != reference on product tree (%s)" % case
        out[case] = {"output": y_ref.clone(), "boxes": bx.clone(), "state_checksum": TS.state_checksum(mine),
                     "weight_seed": 1234, "input_seed": 42}
        print("%-24s ok  out %s  range [%.4f, %.4f]  (%.1fs)" % (case, tuple(y_ref.shape), float(y_ref.min()),
                                                                  float(y_ref.max()), time.time() - t0), flush=True)
    torch.save(out, os.path.join(GOLD, "detection.pt"))


def gen_lowering():
    """The plans lowered from the reference's own model objects: module tree (path, class name), output shape, op
    names and kernel-kind counts for each model, on zero inputs (the lowering reads shapes and module types only)."""
    import pytorchvideo.models.hub as RH
    from pytorchvideo_b200 import testing as TS
    from pytorchvideo_b200.engine.lower import lower_only
    out = {}
    for name, shape in (("x3d_xs", (1, 3, 4, 160, 160)), ("slowfast_r50", (1, 3, 32, 224, 224)),
                        ("mvit_base_16x4", (1, 3, 16, 224, 224))):
        ref = getattr(RH, name)(pretrained=False).eval()
        inp = TS.slowfast_inputs(torch.zeros(shape)) if name.startswith("slowfast") else torch.zeros(shape)
        plan, out_shape = lower_only(ref, inp)
        out[name] = {"input_shapes": [tuple(t.shape) for t in inp] if isinstance(inp, list) else [tuple(inp.shape)],
                     "modules": [(n, type(m).__name__) for n, m in ref.named_modules()],
                     "output_shape": tuple(out_shape), "ops": [n for n, _ in plan.ops], "stats": dict(plan.stats)}
        print("lowering %-16s ok  %d modules, %d ops, out %s" % (name, len(out[name]["modules"]), len(plan.ops),
                                                                  out[name]["output_shape"]), flush=True)
    torch.save(out, os.path.join(GOLD, "lowering.pt"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    ap.add_argument("--skip-models", action="store_true")
    ap.add_argument("--skip-transforms", action="store_true")
    ap.add_argument("--skip-layers", action="store_true")
    ap.add_argument("--skip-detection", action="store_true")
    ap.add_argument("--skip-lowering", action="store_true")
    a = ap.parse_args()
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    if not a.skip_transforms:
        gen_transforms()
    if not a.skip_layers and not a.only:
        gen_layers()
    if not a.skip_detection and not a.only:
        gen_detection()
    if not a.skip_lowering and not a.only:
        gen_lowering()
    if not a.skip_models:
        gen_models(a.only)
