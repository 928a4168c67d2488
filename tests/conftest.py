import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
GOLDEN = ROOT / "tests" / "golden"

torch.set_grad_enabled(False)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def load(name):
        if name not in cache:
            cache[name] = dict(np.load(GOLDEN / f"{name}.npz"))
        return cache[name]

    return load


def lg_pair_from_source(golden, src):
    """'sp_real:api:0:1' -> (kpts0 [N,2] f32, desc0 [256,N], kpts1, desc1) numpy."""
    f, conf, i, j = str(src).split(":")
    b = golden(f)
    return (b[f"{conf}/{i}/keypoints"].astype(np.float32), b[f"{conf}/{i}/descriptors"],
            b[f"{conf}/{j}/keypoints"].astype(np.float32), b[f"{conf}/{j}/descriptors"])


def compressed_descriptors(d, input_proj_w):
    """[256,N] SuperPoint descriptors -> [N,128] unit rows through the orthonormal compression Q = input_proj_w^T
    ([128,256]) of the lg_proj / lg_so fixtures.  Computed in float64 and rounded once to float32, so that every machine
    derives the same inputs."""
    c = np.asarray(input_proj_w, np.float64).T @ np.asarray(d, np.float64)
    c /= np.linalg.norm(c, axis=0, keepdims=True)
    return np.ascontiguousarray(c.T.astype(np.float32))


def match_f1(m_test, m_ref):
    """F1 of the (i, matches0[i]) sets (SURVEY.md 8(d))."""
    a = {(i, int(j)) for i, j in enumerate(np.asarray(m_test)) if j > -1}
    b = {(i, int(j)) for i, j in enumerate(np.asarray(m_ref)) if j > -1}
    if not a and not b:
        return 1.0
    tp = len(a & b)
    return 2 * tp / max(len(a) + len(b), 1)


def assert_keypoints_equivalent(k, s, d, gk, gs, gd, score_tol=1e-3, desc_tol=1e-3, order_noise=2e-5, what="", desc_cols=None):
    """Keypoint parity with the reference (SURVEY.md 8(d)): identical keypoint SET (integer pixel
    coordinates, bit-exact), per-keypoint scores / descriptors within tolerance, and identical ORDER
    up to swaps between keypoints whose reference scores differ by less than the fp32 accumulation
    noise of the conv stack (top-k order is a sort on fp32 scores: bit-identical order would need
    bit-identical scores, which even the reference does not give across devices/BLAS back ends).
    k [N,2] int, s [N], d [256,N].  desc_cols: gd holds only these columns of the reference descriptors."""
    k, gk = np.asarray(k).astype(np.int64), np.asarray(gk).astype(np.int64)
    assert k.shape == gk.shape, f"{what}: {k.shape} vs {gk.shape} keypoints"
    key = lambda a: a[:, 1] * 100000 + a[:, 0]
    a, b = key(k), key(gk)
    lost, gained = np.setdiff1d(b, a), np.setdiff1d(a, b)
    assert len(lost) == 0 and len(gained) == 0, f"{what}: keypoint set differs: lost {len(lost)} gained {len(gained)} of {len(b)}"
    # position of every one of our keypoints in the reference order
    order = {v: i for i, v in enumerate(b.tolist())}
    perm = np.array([order[v] for v in a.tolist()])
    np.testing.assert_allclose(np.asarray(s), np.asarray(gs)[perm], atol=score_tol, err_msg=what)
    if desc_cols is None:
        np.testing.assert_allclose(np.asarray(d), np.asarray(gd)[:, perm], atol=desc_tol, err_msg=what)
    else:
        ours = np.empty_like(perm)
        ours[perm] = np.arange(len(perm))
        np.testing.assert_allclose(np.asarray(d)[:, ours[np.asarray(desc_cols)]], np.asarray(gd), atol=desc_tol, err_msg=what)
    moved = np.nonzero(perm != np.arange(len(perm)))[0]
    if len(moved):
        gs = np.asarray(gs)
        # an element may only move within a run of reference scores that are equal up to the noise
        assert np.all(np.abs(gs[perm[moved]] - gs[moved]) <= order_noise), \
            f"{what}: order differs beyond score noise (max {np.abs(gs[perm[moved]] - gs[moved]).max():.3g})"
    return len(moved)
