"""Three-way gate on the B200 (SURVEY.md §8c): our kernels vs THE REFERENCE'S OWN CUDA kernels, rebuilt for sm_100a
by baseline/build_ref_gpu.py and run on a B200 by tests/golden/make_golden.py --reference-gpu, which records their
outputs for the cases below in tests/golden/reference_gpu.npz.

* vs the -fmad=false build: the pixel planes (RGBA, softmax sum/max, hard depth/face-id) are BIT-EXACT --
  same IEEE operation sequence, same device expf; p2f / gradients differ only by float-atomics order.
* vs the default (FMA-contracted) build only the hard face-index plane is stable (App. B-15): at most a
  handful of mismatching pixels, the rest is reported by tools/ref_gpu_compare.py, not gated.
"""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import ref_gpu_compare as rc  # noqa: E402
from umr_b200 import raster  # noqa: E402
from util import GOLDEN, assert_exact, golden_sample  # noqa: E402

pytestmark = pytest.mark.gpu
KW = dict(sigma_val=1e-5, dist_eps=1e-10, gamma_val=1e-4, anti_aliasing=True)
REFERENCE_GPU = os.path.join(GOLDEN, "reference_gpu.npz")

# Cases run through the reference's -fmad=false build.
# key: (batch, tex_res, seed, icosphere subdiv, image_size, rgb_name, rgb, compare grad_textures)
CASES = {"is128_%s_t%d" % (n, r): (2, r, 5, 3, 128, n, c, False) for n, c in (("softmax", 1), ("hard", 0)) for r in (1, 3)}
# BASELINE config 2 per-image shape: F=1280, 256^2 (S=512), T^2=36, B=2
CASES.update({"c2_%s" % n: (2, 6, 3, 3, 256, n, c, False) for n, c in (("softmax", 1), ("hard", 0))})
# BASELINE config 5 per-image shape: F=5120 (icosphere subdiv 4), 1024^2 (S=2048), B=1.  T^2 == 1: the reference's
# texel-gradient UB (App. B-1) coincides with the intended semantics, so grad_textures is compared too.
CASES.update({"c5_softmax_t1": (1, 1, 9, 4, 1024, "softmax", 1, True), "c5_hard_t2": (1, 2, 9, 4, 1024, "hard", 0, False)})
# Face-index plane of the reference's default (FMA-contracted) build: (batch, tex_res, seed, image_size)
FMA_FACE_INDEX = (2, 2, 6, 128)


def inputs(key):
    """Seeded face vertices, textures and image gradient of a case, on the GPU."""
    B, tex_res, seed, subdiv, IS = CASES[key][:5]
    fv, tex = rc.scene(B, tex_res, seed=seed, subdiv=subdiv)
    g = torch.randn(B, 4, IS, IS, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    return fv, tex, g


def _three_way(key, tex_requires_grad):
    B, tex_res, seed, subdiv, IS, rgb_name, rgb, check_tex_grad = CASES[key]
    z = np.load(REFERENCE_GPU)
    fv, tex, g = inputs(key)
    a = fv.clone().requires_grad_(True)
    t = tex.clone().requires_grad_(tex_requires_grad)
    img, p2f, aggr = raster.soft_rasterize(a, t, IS, aggr_func_rgb=rgb_name, **KW)
    img.backward(g)
    assert_exact(z, key + "/images", img)          # pooled RGBA
    assert_exact(z, key + "/aggrs", aggr)          # aggregation planes
    got, ref = golden_sample(z, key + "/p2f", p2f, 1e-4, 1e-6)
    assert np.allclose(got, ref, rtol=1e-4, atol=1e-6)
    grads = [("grad_faces", a.grad)] + ([("grad_textures", t.grad)] if check_tex_grad else [])
    for name, grad in grads:
        scale = float(z["%s/%s.absmax" % (key, name)])
        got, ref = golden_sample(z, "%s/%s" % (key, name), grad, 1e-3, 1e-5 * scale)
        assert np.allclose(got, ref, rtol=1e-3, atol=1e-5 * scale), name


@pytest.mark.parametrize("rgb_name,rgb", [("softmax", 1), ("hard", 0)])
@pytest.mark.parametrize("tex_res", [1, 3])
def test_bit_exact_with_reference_cuda_kernels_built_without_fma(rgb_name, rgb, tex_res):
    _three_way("is128_%s_t%d" % (rgb_name, tex_res), False)


@pytest.mark.parametrize("tile", [16, 32])
@pytest.mark.parametrize("rgb_name,rgb", [("softmax", 1), ("hard", 0)])
def test_bit_exact_at_c2_shape(rgb_name, rgb, tile, monkeypatch):
    """BASELINE config 2 per-image shape: F=1280, 256^2 (S=512), T^2=36, B=2 -- through both forward kernels."""
    monkeypatch.setattr(raster, "FORWARD_TILE", tile)
    _three_way("c2_%s" % rgb_name, True)


@pytest.mark.parametrize("rgb_name,rgb,tex_res", [("softmax", 1, 1), ("hard", 0, 2)])
def test_bit_exact_at_c5_shape(rgb_name, rgb, tex_res):
    """BASELINE config 5 per-image shape: F=5120 (icosphere subdiv 4), 1024^2 (S=2048), B=1 -- the only shape
    where the cull boxes span several staging pieces and tiles carry long face lists."""
    _three_way("c5_%s_t%d" % (rgb_name, tex_res), True)   # the recorded grad_faces shape pins F = 5120


def test_face_index_plane_against_reference_as_normally_compiled():
    B, tex_res, seed, IS = FMA_FACE_INDEX
    fv, tex = rc.scene(B, tex_res, seed=seed)
    _, _, aggr = raster.soft_rasterize(fv, tex, IS, aggr_func_rgb="hard", **KW)
    ref = torch.from_numpy(np.load(REFERENCE_GPU)["fma/face_index"].astype(np.float32)).cuda()
    assert ref.shape == aggr[:, 1].shape
    mism = int((aggr[:, 1] != ref).sum())
    print("face-id mismatches vs FMA-compiled reference: %d / %d" % (mism, aggr[:, 1].numel()))
    assert mism <= 8  # exact ties / sliver faces only (App. B-15)
