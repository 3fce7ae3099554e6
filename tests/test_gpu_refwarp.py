"""Pins the warp against the REFERENCE ITSELF: outputs of the reference's own CUDA kernel (stnbdhw/BilinearSamplerBDHW.cu:48-109,
compiled for sm_100a by oracle/Makefile, original (32,16) block / (C, H*ceil(W/512), B) grid), recorded on a B200 by
tests/golden/make_warp_golden.py, vs the product's fav_bilinear_sampler_bdhw_update_output / fused temporal input and vs
the C oracle.  Bar: BIT-EXACT at every BASELINE.json config shape, real and stress flows, and on the committed vectors."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_warp_golden  # noqa: E402


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(ROOT, "tests", "golden", "warp_ref_shapes.npz"))


def _ulp_diff(a, b):
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia); ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return int(np.abs(ia - ib).max())


def _assert_reference_output(gold, key, got):
    """got (float32, any shape) equals the reference kernel's output recorded under key, bit for bit."""
    s, want = make_warp_golden.sample(got), gold[key + "_sample"]
    if not np.array_equal(s, want):
        pytest.fail(f"{key}: {int((s != want).sum())} of {s.size} sampled values differ, max ulp {_ulp_diff(want, s)}")
    assert make_warp_golden.digest(got) == str(gold[key + "_sha256"]), f"{key}: differs outside the sampled values"


@pytest.mark.parametrize("shape", make_warp_golden.SHAPES)
def test_product_warp_equals_reference_kernel(gold, shape):
    from fav_b200 import utils

    H, W = shape
    img, flows = make_warp_golden.shape_inputs(H, W)
    img = T(img)
    for name, flow in flows.items():
        g = utils.warp_image(img, T(flow))
        _assert_reference_output(gold, f"{H}x{W}_{name}", g.cpu().numpy())


def test_reference_kernel_batch_channels_and_output_size(gold):
    from fav_b200 import stn

    img, grid, sentinel = make_warp_golden.batch_inputs()
    img, grid = T(img), T(grid)
    assert np.array_equal(gold["batch"], stn.BilinearSamplerBDHW().forward((img, grid)).cpu().numpy())
    assert float(np.abs(gold["sentinel"]).max()) == 0.0  # sentinel flow of vr_helper.lua:10
    assert np.array_equal(gold["sentinel"], stn.BilinearSamplerBDHW().forward((img[:1], T(sentinel))).cpu().numpy())


def test_fused_temporal_input_prior_equals_reference_kernel_composition(gold):
    """in[3:6] of the fused kernel == preprocess(reference-kernel warp) * cert composed with torch ops in the
    reference's op order (core.lua:166-167), bit for bit."""
    from fav_b200 import _lib

    H, W = make_warp_golden.PRIOR_SHAPE
    c, p, flow, cert = (T(a) for a in make_warp_golden.prior_inputs())
    out = torch.empty((7, H, W), device="cuda")
    _lib.check(_lib.lib.fav_temporal_input(_lib.dptr(c), _lib.dptr(p), _lib.dptr(flow), _lib.dptr(cert), None, None,
                                           _lib.dptr(out), H, W, 0, _lib.stream_ptr()))
    _assert_reference_output(gold, "prior", out[3:6].cpu().numpy())


def test_oracle_and_product_reproduce_committed_reference_vectors():
    """tests/golden/warp_ref.npz was written by the reference kernel on a B200 (make_warp_golden.py)."""
    from fav_b200 import stn
    from oracle import pyoracle

    gold = np.load(os.path.join(ROOT, "tests", "golden", "warp_ref.npz"))
    for case in make_warp_golden.WARP_CASES:
        img, flow = make_warp_golden.warp_inputs(case)
        assert np.array_equal(stn.BilinearSamplerBDHW().forward((T(img), T(flow))).cpu().numpy(), gold[case[0]]), case[0]
        assert np.array_equal(pyoracle.warp_bdhw(img, flow), gold[case[0]]), case[0]
