"""The torch layout helpers of tests/util.py (used on the device by test_kernels_at_scale_gpu.py) against the
NumPy planes emulation and the flattened-feature layout, on small ragged shapes; runs without a GPU."""
import numpy as np
import pytest
import torch

from util import Geo, dropout_mask, dropout_mask_t, from_feat_t, from_planes, from_planes_t, to_feat_t, to_planes, to_planes_t


@pytest.mark.parametrize('seed,draw,keep', [(0, 0, 0.5), (12345, 7, 0.75), (0xFFFFFFFF, 0xDEADBEEF, 0.1)])
def test_torch_dropout_mask_equals_the_numpy_restatement(seed, draw, keep):
    shape = (3, 5, 7, 16)
    ref = dropout_mask(seed, draw, shape, keep)
    got = dropout_mask_t(seed, draw, shape, keep, 'cpu')
    np.testing.assert_array_equal(got.numpy().astype(np.float32), ref)
    assert 0 < ref.mean() < 1


@pytest.mark.parametrize('B,H,W,C,Cpad', [(1, 4, 4, 8, None), (3, 8, 8, 3, 16), (5, 4, 6, 24, None), (2, 32, 32, 16, 32),
                                          (7, 2, 2, 13, 16)])
def test_planes_helpers_equal_the_numpy_layout(B, H, W, C, Cpad):
    rng = np.random.default_rng(B * 100 + H)
    x = rng.standard_normal((B, H, W, C)).astype(np.float32)
    geo = Geo(B, H, W)
    ref = to_planes(x, geo, Cpad)
    got = to_planes_t(torch.from_numpy(x), geo, Cpad)
    assert got.dtype == torch.float32 and tuple(got.shape) == ref.shape
    np.testing.assert_array_equal(got.numpy(), ref)
    np.testing.assert_array_equal(from_planes_t(got, geo, C).numpy(), from_planes(ref, geo, C))
    np.testing.assert_array_equal(from_planes_t(got, geo, C).numpy(), x)
    # dtype follows the input, and a bf16 round trip is the identity on bf16 values
    xb = torch.from_numpy(x).to(torch.bfloat16)
    tb = to_planes_t(xb, geo, Cpad)
    assert tb.dtype == torch.bfloat16
    assert torch.equal(from_planes_t(tb, geo, C), xb)


@pytest.mark.parametrize('B,F,Balloc', [(1, 8, 8), (5, 256, 8), (37, 64, 128), (129, 40, 256)])
def test_feature_helpers_equal_the_loop_layout(B, F, Balloc):
    rng = np.random.default_rng(F + B)
    x = rng.standard_normal((B, F)).astype(np.float32)
    ref = np.zeros((F // 8, Balloc, 8), np.float32)
    for i in range(F // 8):                       # the layout as test_kernels_gpu.py builds it
        ref[i, :B] = x[:, i * 8:(i + 1) * 8]
    got = to_feat_t(torch.from_numpy(x), Balloc)
    np.testing.assert_array_equal(got.numpy(), ref)
    np.testing.assert_array_equal(from_feat_t(got, B).numpy(), np.concatenate([ref[i, :B] for i in range(F // 8)], 1))
