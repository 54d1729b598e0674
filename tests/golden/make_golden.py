"""Generate the committed golden fixtures from THE REFERENCE ITSELF.

    python tests/golden/make_golden.py                    # needs the reference's sources (oracle A)
    python tests/golden/make_golden.py --reference-gpu [--out DIR]   # needs baseline/_ref/*.so and a B200

Without arguments it runs oracle A = the reference's own rasteriser device code compiled for the host
(oracle/ref_host_shim.cpp) and writes
* one .npz per entry of CASES with the seeded inputs and the reference's outputs, small enough to commit.
  grad_textures is stored only for T2 == 1, where the reference's undefined behaviour (kernel.cu:199-218) cannot
  matter; for T2 > 1 it is pinned by finite differences in tests/test_oracle.py instead;
* reference_host.npz: oracle A's outputs for the cases of tests/test_oracle.py that compare oracle B with it.
With --reference-gpu it runs the reference's own CUDA kernels rebuilt for sm_100a (baseline/build_ref_gpu.py) on
the cases of tests/test_reference_gpu.py and writes reference_gpu.npz.
The two reference_*.npz files keep compact records (tests/util.py): SHA-256 digests of the outputs compared bit for
bit, fixed samples plus max |value| and L2 norm of those compared within a tolerance.
Deterministic: single-threaded host runs (float atomics order).
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from util import record_close, record_exact  # noqa: E402

CASES = {
    # name: (B, subdiv, tex_res, image_size, aa, rgb, seed)
    "softmax_aa_t1": (1, 2, 1, 32, True, "softmax", 11),
    "softmax_aa_t4": (2, 2, 2, 24, True, "softmax", 12),
    "hard_aa_t4": (1, 2, 2, 32, True, "hard", 13),
    "softmax_noaa_t9": (1, 1, 3, 40, False, "softmax", 14),
    "hard_noaa_t1": (1, 2, 1, 48, False, "hard", 15),
}


def _save(path, rec):
    np.savez_compressed(path, **rec)
    print(os.path.basename(path), os.path.getsize(path), "bytes")


def vectors(out):
    import softras
    from util import scene
    for name, (B, sd, tr, isz, aa, rgb, seed) in CASES.items():
        fv, tex = scene(B, sd, tr, seed)
        img, fwd, cfg = softras.render(fv, tex, isz, anti_aliasing=aa, impl="A", nthreads=1, aggr_func_rgb=rgb,
                                       sigma_val=1e-5, dist_eps=1e-10, gamma_val=1e-4)
        g = np.random.default_rng(seed + 100).normal(size=img.shape).astype(np.float32)
        gf, gt = softras.render_backward(fwd, cfg, g, anti_aliasing=aa, impl="A", nthreads=1)
        rec = dict(face_vertices=fv, textures=tex, grad_images=g, images=img, aggrs_info=fwd["aggrs_info"],
                   p2f_info=fwd["p2f_info"], grad_faces=gf, image_size=isz, anti_aliasing=aa, rgb=rgb)
        if tr == 1:
            rec["grad_textures"] = gt
        _save(os.path.join(out, name + ".npz"), rec)


def reference_host(out):
    import test_oracle as T
    rec = {}
    for rgb, aa, isz, tr in T.BIT_EXACT_CASES:
        for k, v in T.bit_exact_case("A", rgb, aa, isz, tr).items():
            record_exact(rec, "bit_exact/%s_%s_%d_%d/%s" % (rgb, aa, isz, tr, k), v)
    for dist, alpha in T.OTHER_MODES:
        for k, v in T.other_modes_case("A", dist, alpha).items():
            record_close(rec, "other_modes/%s_%s/%s" % (dist, alpha, k), v)
    for seed in T.RANDOMISED_SEEDS:
        for k, v in T.randomised_case("A", seed)[0].items():
            record_exact(rec, "randomised/%d/%s" % (seed, k), v)
    _save(os.path.join(out, "reference_host.npz"), rec)


def reference_gpu(out):
    import torch.nn.functional as F
    import test_reference_gpu as T
    rc = T.rc
    nofma, fma = rc.load("soft_rasterize_ref_nofma"), rc.load("soft_rasterize_ref")
    assert nofma is not None and fma is not None, "build baseline/_ref first: python baseline/build_ref_gpu.py [--no-fma]"
    rec = {}
    for key, (B, tex_res, seed, subdiv, IS, rgb_name, rgb, tex_grad) in T.CASES.items():
        fv, tex, g = T.inputs(key)
        S = 2 * IS
        colors, p2f, aggrs, finfo = rc.ref_forward(nofma, fv, tex, S, rgb)
        ghi = (g / 4).repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)
        gf, gt = rc.ref_backward(nofma, fv, tex, colors, finfo, aggrs, ghi, S, rgb)
        record_exact(rec, key + "/images", F.avg_pool2d(colors, 2, 2).cpu().numpy())
        record_exact(rec, key + "/aggrs", aggrs.cpu().numpy())
        record_close(rec, key + "/p2f", p2f.cpu().numpy())
        record_close(rec, key + "/grad_faces", gf.cpu().numpy())
        if tex_grad:
            record_close(rec, key + "/grad_textures", gt.cpu().numpy())
    B, tex_res, seed, IS = T.FMA_FACE_INDEX
    fv, tex = rc.scene(B, tex_res, seed=seed)
    face = rc.ref_forward(fma, fv, tex, 2 * IS, 0)[2][:, 1].cpu().numpy()
    rec["fma/face_index"] = face.astype(np.int16)
    assert np.array_equal(rec["fma/face_index"], face)
    _save(os.path.join(out, "reference_gpu.npz"), rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference-gpu", action="store_true")
    ap.add_argument("--out", default=HERE)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    if args.reference_gpu:
        reference_gpu(args.out)
        return
    import softras
    assert softras.have_oracle_a(), "oracle A (reference on host) is required to (re)generate goldens"
    vectors(args.out)
    reference_host(args.out)


if __name__ == "__main__":
    main()
