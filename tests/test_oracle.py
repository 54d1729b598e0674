"""CPU tests of the oracle (no GPU): oracle B (our restatement) is pinned
(1) bit-exactly against oracle A = the reference's own device code compiled for the host, through its outputs
    recorded in tests/golden/reference_host.npz (tests/golden/make_golden.py runs the same cases through oracle A),
(2) against the committed golden vectors generated from oracle A (tests/golden/make_golden.py),
(3) by finite differences for the one deliberate difference (texel gradient, App. B-1),
(4) by domain invariants."""
import glob
import os

import numpy as np
import pytest

import softras
from util import GOLDEN as GOLDEN_DIR, assert_exact, golden_sample, rel_report, scene

GOLDEN = sorted(glob.glob(os.path.join(GOLDEN_DIR, "*_t[0-9].npz")))
REFERENCE_HOST = os.path.join(GOLDEN_DIR, "reference_host.npz")
UMR = dict(sigma_val=1e-5, dist_eps=1e-10, gamma_val=1e-4)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_b_matches_golden_vectors(path):
    z = np.load(path)
    isz, aa, rgb = int(z["image_size"]), bool(z["anti_aliasing"]), str(z["rgb"])
    img, fwd, cfg = softras.render(z["face_vertices"], z["textures"], isz, anti_aliasing=aa, impl="B", nthreads=1,
                                   aggr_func_rgb=rgb, **UMR)
    gf, gt = softras.render_backward(fwd, cfg, z["grad_images"], anti_aliasing=aa, impl="B", nthreads=1)
    # single-threaded, same op order: bit-exact with the reference-as-compiled
    assert np.array_equal(img, z["images"])
    assert np.array_equal(fwd["aggrs_info"], z["aggrs_info"])
    assert np.array_equal(fwd["p2f_info"], z["p2f_info"])
    assert np.array_equal(gf, z["grad_faces"])
    if "grad_textures" in z.files:
        assert np.array_equal(gt, z["grad_textures"])


BIT_EXACT_CASES = [(rgb, aa, isz, tr) for aa, isz, tr in [(True, 32, 2), (False, 50, 1)] for rgb in ["softmax", "hard"]]
RANDOMISED_SEEDS = range(8)
OTHER_MODES = [("barycentric", "sum"), ("hard", "hard"), ("euclidean", "sum")]


def bit_exact_case(impl, rgb, aa, isz, tr):
    """Outputs of one render + backward through oracle `impl`; make_golden.py records them for impl="A"."""
    fv, tex = scene(2, 3, tr, seed=21)
    img, fwd, cfg = softras.render(fv, tex, isz, anti_aliasing=aa, impl=impl, nthreads=1, aggr_func_rgb=rgb, **UMR)
    g = np.random.default_rng(5).normal(size=img.shape).astype(np.float32)
    gf, gt = softras.render_backward(fwd, cfg, g, anti_aliasing=aa, impl=impl, nthreads=1)
    out = {k: fwd[k] for k in ("soft_colors", "aggrs_info", "faces_info", "p2f_info")}
    out.update(images=img, grad_faces=gf)
    if tr == 1:  # T2 == 1: the reference's UB cannot matter
        out["grad_textures"] = gt
    return out


def other_modes_case(impl, dist, alpha):
    fv, tex = scene(1, 2, 1, seed=22)
    cfg = softras.RasterCfg(48, dist_func=dist, aggr_func_alpha=alpha, dist_eps=1e-4, sigma_val=1e-4)
    fwd = softras.forward(fv, tex, cfg, impl=impl, nthreads=1)
    g = np.random.default_rng(6).normal(size=fwd["soft_colors"].shape).astype(np.float32)
    gf, _ = softras.backward(fwd, g, cfg, impl=impl, nthreads=1)
    return dict(soft_colors=fwd["soft_colors"], aggrs_info=fwd["aggrs_info"], grad_faces=gf)


@pytest.mark.parametrize("rgb", ["softmax", "hard"])
@pytest.mark.parametrize("aa,isz,tr", [(True, 32, 2), (False, 50, 1)])
def test_oracle_b_bit_exact_with_reference_on_host(rgb, aa, isz, tr):
    z = np.load(REFERENCE_HOST)
    for k, v in bit_exact_case("B", rgb, aa, isz, tr).items():
        assert_exact(z, "bit_exact/%s_%s_%d_%d/%s" % (rgb, aa, isz, tr, k), v)


def test_other_modes_match_reference_on_host():
    """Modes UMR does not use (barycentric / hard distance, sum / hard alpha): restated too."""
    z = np.load(REFERENCE_HOST)
    for dist, alpha in OTHER_MODES:
        for k, v in other_modes_case("B", dist, alpha).items():
            key = "other_modes/%s_%s/%s" % (dist, alpha, k)
            got, ref = golden_sample(z, key, v, 1e-6, 1e-7)
            ok, msg = rel_report(key, got, ref, 1e-6, 1e-7)
            assert ok, msg


def test_texel_gradient_matches_finite_differences():
    """Intended semantics of kernel.cu:199-218 (only the sampled texel gets gradient): the render is
    linear in the texels, so central differences in float64 are exact up to rounding."""
    fv, tex = scene(1, 1, 2, seed=23)
    cfg = softras.RasterCfg(24, **UMR)
    fv64, tex64 = fv.astype(np.float64), tex.astype(np.float64)
    fwd = softras.forward(fv64, tex64, cfg, impl="B", nthreads=1, dtype=np.float64)
    g = np.random.default_rng(7).normal(size=fwd["soft_colors"].shape)
    _, gt = softras.backward(fwd, g, cfg, impl="B", nthreads=1)
    _, gt_ub = softras.backward(fwd, g, cfg, impl="B", ub_texgrad=True, nthreads=1)
    idx = np.argwhere(np.abs(gt) > 1e-3)[:6]
    assert len(idx) > 0
    for b, f, t, k in idx:
        fd = []
        for s in (+1e-3, -1e-3):
            tx = tex64.copy()
            tx[b, f, t, k] += s
            o = softras.forward(fv64, tx, cfg, impl="B", nthreads=1, dtype=np.float64)
            fd.append((o["soft_colors"] * g).sum())
        num = (fd[0] - fd[1]) / 2e-3
        assert abs(num - gt[b, f, t, k]) <= 1e-6 * max(1.0, abs(num)), (num, gt[b, f, t, k])
    # the as-compiled behaviour smears the face total over every texel: strictly larger support
    assert (np.abs(gt_ub) > 0).sum() > (np.abs(gt) > 0).sum()


def test_vertex_gradient_matches_finite_differences_in_z():
    """dL/dz is exact in the reference formulation (SURVEY.md App. C); x/y gradients deliberately ignore
    the cull / w_clip dependence so they are not FD-checkable at UMR's sigma."""
    fv, tex = scene(1, 1, 2, seed=24)
    cfg = softras.RasterCfg(24, **UMR)
    fv64, tex64 = fv.astype(np.float64), tex.astype(np.float64)
    fwd = softras.forward(fv64, tex64, cfg, impl="B", nthreads=1, dtype=np.float64)
    g = np.zeros_like(fwd["soft_colors"])
    g[:, :3] = np.random.default_rng(8).normal(size=g[:, :3].shape)
    gf, _ = softras.backward(fwd, g, cfg, impl="B", nthreads=1)
    zs = np.argsort(-np.abs(gf[0, :, 2::3]).ravel())[:4]
    for j in zs:
        f, c = divmod(int(j), 3)
        num = []
        for s in (+1e-6, -1e-6):
            x = fv64.copy()
            x[0, f, 3 * c + 2] += s
            o = softras.forward(x, tex64, cfg, impl="B", nthreads=1, dtype=np.float64)
            num.append((o["soft_colors"] * g).sum())
        fd = (num[0] - num[1]) / 2e-6
        assert abs(fd - gf[0, f, 3 * c + 2]) <= 1e-4 * max(abs(fd), 1e-6), (fd, gf[0, f, 3 * c + 2])


def test_invariants():
    fv, tex = scene(2, 3, 2, seed=25)
    img, fwd, _ = softras.render(fv, tex, 32, impl="B", **UMR)
    a = fwd["soft_colors"][:, 3]
    assert a.min() >= 0 and a.max() <= 1
    rgb = fwd["soft_colors"][:, :3]
    assert rgb.min() >= -1e-6 and rgb.max() <= 1 + 1e-5      # convex combination of texels and bg (0)
    imgh, fwdh, _ = softras.render(fv, tex, 32, impl="B", aggr_func_rgb="hard", **UMR)
    fid = fwdh["aggrs_info"][:, 1]
    assert ((fid >= -1) & (fid < fv.shape[1]) & (fid == np.round(fid))).all()
    assert ((fid >= 0) == (fwdh["aggrs_info"][:, 0] < 1e7)).all()
    assert np.abs(fwdh["p2f_info"]).max() == 0                 # hard mode never accumulates p2f (B-4)
    # mirrored mesh (x -> -x, which flips the winding: double-sided rendering) => mirrored silhouette
    fvm = fv.copy()
    fvm[:, :, 0::3] *= -1
    _, fwdm, _ = softras.render(fvm, tex, 32, impl="B", **UMR)
    ok, msg = rel_report("mirror alpha", fwdm["soft_colors"][:, 3][:, :, ::-1], a, 1e-4, 1e-5)
    assert ok, msg


def test_empty_and_degenerate_inputs():
    fv, tex = scene(1, 1, 1, seed=26)
    fv_far = fv.copy()
    fv_far[:, :, 0::3] += 10.0                                  # everything off-screen
    img, fwd, _ = softras.render(fv_far, tex, 16, impl="B", **UMR)
    assert np.abs(img).max() == 0 and np.abs(fwd["p2f_info"]).max() == 0
    fv_deg = fv.copy()
    fv_deg[0, 0, 3:6] = fv_deg[0, 0, 0:3]                       # zero-area triangle: det clamp path
    fv_deg[0, 1, :] = np.tile(fv_deg[0, 1, 0:3], 3)
    img, _, _ = softras.render(fv_deg, tex, 16, impl="B", **UMR)
    assert np.isfinite(img).all()


def randomised_case(impl, seed):
    rng = np.random.default_rng(1000 + seed)
    B = int(rng.integers(1, 3))
    subdiv = int(rng.integers(0, 3))
    S = int(rng.integers(9, 70))
    tex_res = int(rng.choice([1, 2, 3]))
    kw = dict(sigma_val=float(10 ** rng.uniform(-5.5, -3.5)), gamma_val=float(10 ** rng.uniform(-4.5, -2)),
              dist_eps=float(10 ** rng.uniform(-10, -3)), near=float(rng.uniform(0.5, 7.5)),
              far=float(rng.uniform(7.8, 100)), fill_back=bool(rng.integers(0, 2)),
              background_color=tuple(float(x) for x in rng.uniform(0, 1, 3)),
              aggr_func_rgb=str(rng.choice(["softmax", "hard"])))
    fv, tex = scene(B, subdiv, tex_res, seed=2000 + seed)
    cfg = softras.RasterCfg(S, **kw)
    fwd = softras.forward(fv, tex, cfg, impl=impl, nthreads=1)
    g = np.random.default_rng(seed).normal(size=fwd["soft_colors"].shape).astype(np.float32)
    gf, gt = softras.backward(fwd, g, cfg, impl=impl, nthreads=1)
    out = {k: fwd[k] for k in ("soft_colors", "aggrs_info", "p2f_info")}
    out["grad_faces"] = gf
    if tex_res == 1:  # reference UB (App. B-1) otherwise
        out["grad_textures"] = gt
    return out, kw


@pytest.mark.parametrize("seed", RANDOMISED_SEEDS)
def test_randomised_configurations_match_reference_on_host(seed):
    """Random sweep over the scalar arguments of soft_rasterize (sizes, softness, clipping planes, culling,
    background): restatement == reference-on-host, bit for bit (single-threaded, T2 == 1 for grad_textures)."""
    z = np.load(REFERENCE_HOST)
    out, kw = randomised_case("B", seed)
    print("configuration:", kw)
    for k, v in out.items():
        assert_exact(z, "randomised/%d/%s" % (seed, k), v)
