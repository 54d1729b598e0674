"""Shared helpers for the parity tests: seeded scenes, tolerance reports and the compact golden records of the
reference's outputs (tests/golden/make_golden.py writes them, the tests read them)."""
import hashlib
import os

import numpy as np

from umr_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE = 1024  # values kept of an array that is compared within a tolerance


def scene(B=2, subdiv=3, tex_res=2, seed=0):
    """Seeded raster-space inputs: face_vertices [B,F,9] f32, textures [B,F,R*R,3] f32."""
    rng = np.random.default_rng(seed)
    v, f = synth.icosphere(subdiv)
    verts = synth.bird_like(v, rng, B)
    cams = synth.cameras(rng, B)
    fv = synth.raster_space_faces(verts, f, cams)
    tex = rng.uniform(0, 1, size=(B, f.shape[0], tex_res * tex_res, 3)).astype(np.float32)
    return fv, tex


def rel_report(name, got, ref, rtol=1e-4, atol=1e-6):
    """Returns (ok, message). ok <=> |got-ref| <= atol + rtol*max(|got|,|ref|) everywhere."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    diff = np.abs(got - ref)
    bound = atol + rtol * np.maximum(np.abs(got), np.abs(ref))
    bad = diff > bound
    nb = int(bad.sum())
    denom = np.linalg.norm(ref.ravel()) + 1e-30
    msg = "%s: max|d|=%.3e rel-L2=%.3e bad=%d/%d (%.4f%%) max|ref|=%.3e" % (
        name, diff.max() if diff.size else 0.0, np.linalg.norm(diff.ravel()) / denom, nb, diff.size,
        100.0 * nb / max(diff.size, 1), np.abs(ref).max() if ref.size else 0.0)
    if nb:
        i = np.unravel_index(np.argmax(diff - bound), diff.shape)
        msg += " worst@%s got=%.9g ref=%.9g" % (str(tuple(int(x) for x in i)), got[i], ref[i])
    return nb == 0, msg


# ---- golden records of the reference's outputs ---------------------------------------------------------------------
# An output compared bit for bit is kept as the SHA-256 of its float32 bytes; one compared within a tolerance as SAMPLE
# values at fixed positions plus its max |value| and L2 norm.  That keeps outputs of megabytes in a few kilobytes.

def sample_index(size, n=SAMPLE):
    """Fixed positions in a flattened array of `size` values: i * p mod size for a prime p, so they are distinct and
    spread over every image, channel and row."""
    if size <= n:
        return np.arange(size)
    return np.arange(n, dtype=np.int64) * 2654435761 % size


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float32).tobytes()).hexdigest()


def record_exact(rec, key, a):
    a = np.asarray(a, dtype=np.float32)
    rec[key + ".shape"] = np.array(a.shape)
    rec[key + ".sha256"] = np.array(sha256(a))


def record_close(rec, key, a):
    a = np.asarray(a, dtype=np.float32)
    rec[key + ".shape"] = np.array(a.shape)
    rec[key + ".sample"] = a.ravel()[sample_index(a.size)]
    rec[key + ".absmax"] = np.array(np.abs(a).max(), np.float64)
    rec[key + ".norm"] = np.array(np.linalg.norm(a.ravel().astype(np.float64)))


def _shape(z, key, got):
    assert tuple(got.shape) == tuple(int(x) for x in z[key + ".shape"]), "%s: shape %s, reference %s" % (
        key, tuple(got.shape), tuple(z[key + ".shape"]))


def assert_exact(z, key, got):
    """`got` (numpy array or tensor) is bit-identical to the recorded reference output `key`."""
    got = np.asarray(got.detach().cpu() if hasattr(got, "detach") else got, dtype=np.float32)
    _shape(z, key, got)
    assert sha256(got) == str(z[key + ".sha256"]), "%s differs from the reference's output" % key


def golden_sample(z, key, got, rtol, atol):
    """Returns (got, reference) at the recorded positions, float64.  Also checks the whole array's L2 norm against the
    reference's, within the bound that |got - ref| <= atol + rtol * max(|got|, |ref|) everywhere implies."""
    got = np.asarray(got.detach().cpu() if hasattr(got, "detach") else got, dtype=np.float64)
    _shape(z, key, got)
    norm, ref_norm = np.linalg.norm(got.ravel()), float(z[key + ".norm"])
    bound = atol * np.sqrt(got.size) + rtol * (norm + ref_norm)
    assert abs(norm - ref_norm) <= bound, "%s: L2 norm %.9g, reference %.9g" % (key, norm, ref_norm)
    return got.ravel()[sample_index(got.size)], z[key + ".sample"].astype(np.float64)
