"""The oracle is pinned before it is trusted (CPU only):
  * checkConsistency / computeCorners restatement == the reference's own consistencyChecker binary, bit for bit,
    on the committed golden masks (tests/golden/consistency_*.npz, written by oracle/_ref), the frame passed in
    memory and through a P6 file;
  * the warp restatement is cross-checked against torch grid_sample (independent implementation of per-corner
    zero fill), min_filter against F.max_pool2d, pre/deprocess against the Lua formula;
  * the torch net oracle reproduces its committed fp64 outputs and agrees fp32 vs fp64.
"""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from fav_b200 import synth
from oracle import net_oracle, pyoracle

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_golden  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.mark.parametrize("case", make_golden.CONSISTENCY_CASES)
def test_consistency_oracle_equals_reference_binary_golden(case):
    H, W, idx, sigma, seed = case
    g = np.load(os.path.join(GOLD, f"consistency_{H}x{W}.npz"))
    ref3 = np.unpackbits(g["ref3"])[: H * W].reshape(H, W).astype(np.uint8) * 255
    ref4 = np.unpackbits(g["ref4"])[: H * W].reshape(H, W).astype(np.uint8) * 255
    bw, fw, _, img255 = make_golden.consistency_inputs(H, W, idx, sigma, seed)
    assert np.array_equal(pyoracle.consistency(bw, fw), ref3)
    assert np.array_equal(pyoracle.consistency(bw, fw, img255), ref4)
    if sigma > 0:
        assert (ref3 != ref4).sum() > 0  # the structure term is actually exercised


def test_consistency_oracle_equals_reference_binary_live(tmp_path):
    """The frame goes through a P6 file and read_ppm_planes, as the binary reads it; the binary's masks on these files
    are tests/golden/consistency_72x88.npz (make_golden.py)."""
    H, W = 72, 88
    g = np.load(os.path.join(GOLD, f"consistency_{H}x{W}.npz"))
    ref3 = np.unpackbits(g["ref3"])[: H * W].reshape(H, W).astype(np.uint8) * 255
    ref4 = np.unpackbits(g["ref4"])[: H * W].reshape(H, W).astype(np.uint8) * 255
    bw, fw, fr, _ = make_golden.consistency_inputs(H, W, 5, 0.5, 11)
    d = str(tmp_path)
    synth.write_ppm(d + "/f.ppm", fr)
    from fav_b200.consistencyChecker import read_ppm_planes

    img = read_ppm_planes(d + "/f.ppm")
    assert np.array_equal(pyoracle.consistency(bw, fw), ref3)
    assert np.array_equal(pyoracle.consistency(bw, fw, img), ref4)


def test_warp_oracle_reproduces_reference_kernel_vectors():
    """tests/golden/warp_ref.npz = outputs of the REFERENCE's own CUDA kernel (stnbdhw/BilinearSamplerBDHW.cu:48-109 compiled
    for sm_100a, oracle/ref_warp) on a B200, written by tests/golden/make_warp_golden.py: the C restatement (including the
    FMA contraction of :103-106) must reproduce them bit for bit -- this pins orc_warp_bdhw with the reference itself."""
    import make_warp_golden

    gold = np.load(os.path.join(GOLD, "warp_ref.npz"))
    for case in make_warp_golden.WARP_CASES:
        img, flow = make_warp_golden.warp_inputs(case)
        assert np.array_equal(pyoracle.warp_bdhw(img, flow), gold[case[0]]), case[0]


def _grid_sample_warp(img, flow):
    C, H, W = img.shape
    y, x = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
    gx = (x + flow[1]) / (W - 1) * 2 - 1
    gy = (y + flow[0]) / (H - 1) * 2 - 1
    grid = torch.from_numpy(np.stack([gx, gy], -1))[None]
    return F.grid_sample(torch.from_numpy(img.astype(np.float64))[None], grid, mode="bilinear", padding_mode="zeros",
                         align_corners=True)[0].numpy()


@pytest.mark.parametrize("shape", [(40, 56), (33, 47)])
def test_warp_oracle_vs_grid_sample(shape):
    H, W = shape
    img = synth.make_frame(H, W, 1)
    flow = synth.checker_to_lua(synth.make_backward_flow(H, W, 2))
    flow[:, :4] += 7.3  # push samples across the border: per-corner zero fill (BilinearSamplerBDHW.cu:92-101)
    o = pyoracle.warp_bdhw(img, flow)
    assert np.abs(o - _grid_sample_warp(img, flow)).max() < 2e-5
    # sentinel flow 99999 (vr_helper.lua:10) must map to exactly 0
    flow[:] = 99999.0
    assert np.all(pyoracle.warp_bdhw(img, flow) == 0)


def test_warp_oracle_shapes_and_batching():
    img = np.random.default_rng(0).uniform(size=(2, 3, 10, 12)).astype(np.float32)
    grid = np.random.default_rng(1).uniform(-3, 3, size=(2, 2, 7, 9)).astype(np.float32)  # out size != in size
    out = pyoracle.warp_bdhw(img, grid)
    assert out.shape == (2, 3, 7, 9)
    assert np.array_equal(pyoracle.warp_bdhw(img[1], grid[1]), out[1])  # 3-D inputs auto-batched (.lua:59-65)
    assert np.array_equal(pyoracle.warp_bdhw(img, grid, threads=4), out)


def test_min_filter_oracle_vs_maxpool():
    rng = np.random.default_rng(3)
    for (H, W, r) in [(20, 31, 7), (9, 9, 3), (5, 40, 7)]:
        x = rng.uniform(0, 1, size=(H, W)).astype(np.float32)
        t = torch.from_numpy(x)[None, None]
        ref = (-(F.max_pool2d(-t + 1, r, 1, r // 2)) + 1)[0, 0].numpy()  # utils.lua:161-169
        assert np.array_equal(pyoracle.min_filter(x, r), ref)


def test_preprocess_roundtrip_and_formula():
    img = synth.make_frame(16, 24, 1)
    pre = pyoracle.vgg_preprocess(img)
    mean = np.array([103.939, 116.779, 123.68], np.float32)
    assert np.array_equal(pre, img[::-1] * np.float32(255) - mean[:, None, None])
    assert np.abs(pyoracle.vgg_deprocess(pre) - img).max() < 1e-6


def test_temporal_input_composition():
    H, W = 24, 40
    c, p = synth.make_frame(H, W, 2), synth.make_frame(H, W, 1)
    flow = synth.checker_to_lua(synth.make_backward_flow(H, W, 2))
    cert = (np.random.default_rng(0).uniform(size=(H, W)) > 0.3).astype(np.float32)
    x7 = pyoracle.temporal_input(c, p, flow, cert)
    assert np.array_equal(x7[:3], pyoracle.vgg_preprocess(c))
    assert np.array_equal(x7[6], cert)
    warped = pyoracle.vgg_preprocess(pyoracle.warp_bdhw(p, flow))
    assert np.array_equal(x7[3:6], warped * cert[None] + 0.0)
    # an out-of-frame sample under certainty 1 is -mean, not 0 (SURVEY appendix A)
    flow2 = np.full_like(flow, 1e4)
    x7b = pyoracle.temporal_input(c, p, flow2, np.ones((H, W), np.float32))
    assert np.allclose(x7b[3:6, 0, 0], [-103.939, -116.779, -123.68])


def test_net_oracle_matches_committed_golden_and_fp32():
    g = np.load(os.path.join(GOLD, "clip_64x96.npz"))["outs"]
    o64 = net_oracle.run_clip(net_oracle.NetOracle(style="candy", dtype=torch.float64), 64, 96, 3)
    assert np.abs(np.stack(o64) - g).max() < 1e-6
    o32 = net_oracle.run_clip(net_oracle.NetOracle(style="candy", dtype=torch.float32), 64, 96, 3)
    assert np.abs(np.stack(o32) - g).max() < 5e-5


def test_net_oracle_structure():
    net = net_oracle.NetOracle()
    assert net.pad == 40  # SpatialReflectionPadding(40,...) for 5 residual blocks at 1/4 resolution
    taps = {}
    net.forward(torch.zeros(1, 7, 48, 64, dtype=torch.float64), taps)
    # appendix B size rule: 48x64 -> 128x144 -> 64x72 -> 32x36 -> (5 res) 12x16 -> 24x32 -> 48x64
    assert tuple(taps["l0"].shape[-2:]) == (128, 144) and tuple(taps["l2"].shape[-2:]) == (32, 36)
    assert tuple(taps["l7"].shape[-2:]) == (12, 16) and tuple(taps["l9"].shape[-2:]) == (48, 64)
