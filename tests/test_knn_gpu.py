"""GPU parity of distCUDA2 (SURVEY.md §8 row f3): this library's kernels (through `simple_knn._C.distCUDA2` -> C ABI)
against the CPU oracle AND against what the original project's own simple_knn.cu, compiled unmodified, returned on the
same clouds (stored under tests/golden/).

Tolerance: the quantity is a float32 sum of three float32 squared distances; implementations differ in FMA contraction
and summation order only -> 1e-6 relative (about 8 ulp), stated here once."""
import os

import numpy as np
import pytest
import torch

import helpers  # noqa: F401
from oracle import knn_oracle

pytestmark = pytest.mark.gpu
RTOL = 1e-6


def _cloud(kind, P, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "ball":            # the reference's own initialisation (gs_renderer.py:694-702)
        phi, ct, r = rng.random(P) * 2 * np.pi, rng.random(P) * 2 - 1, 0.5 * np.cbrt(rng.random(P))
        st = np.sqrt(1 - ct * ct)
        p = np.stack([r * st * np.cos(phi), r * st * np.sin(phi), r * ct], axis=1)
    elif kind == "clusters":
        p = rng.normal(size=(P, 3)) * 0.003 + rng.integers(0, 7, (P, 1)) * np.array([[1.0, -2.0, 0.5]])
    elif kind == "plane":
        p = np.concatenate([rng.random((P, 2)), np.zeros((P, 1))], axis=1)
    elif kind == "line":
        p = np.concatenate([np.zeros((P, 1)), rng.random((P, 1)) * 3, np.full((P, 1), 0.25)], axis=1)
    elif kind == "duplicates":
        base = rng.random((P // 4, 3))
        p = np.concatenate([base, base, base, rng.random((P - 3 * (P // 4), 3))], axis=0)
    elif kind == "surface":       # points on a sphere shell: empty interior, very uneven cells
        v = rng.normal(size=(P, 3)); p = v / np.linalg.norm(v, axis=1, keepdims=True)
    else:
        raise ValueError(kind)
    return np.ascontiguousarray(p.astype(np.float32))


def _ours(p):
    from simple_knn._C import distCUDA2          # the import the reference makes (gs_renderer.py:14)
    return distCUDA2(torch.tensor(p, device="cuda")).cpu().numpy()


@pytest.mark.parametrize("kind,P", [("ball", 5000), ("ball", 100000), ("clusters", 30000), ("plane", 20000), ("line", 5000),
                                    ("duplicates", 8000), ("surface", 50000)])
def test_matches_the_cpu_oracle(kind, P):
    p = _cloud(kind, P)
    ref = knn_oracle.dist2_f64(p)
    got = _ours(p)
    np.testing.assert_allclose(got, ref, rtol=RTOL, atol=1e-30)


REF_CASES = [("ball", 100000), ("clusters", 30000), ("plane", 20000), ("duplicates", 8000), ("surface", 50000)]
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "simple_knn_vectors.npz")


@pytest.mark.parametrize("kind,P", REF_CASES)
def test_matches_the_reference_implementation_itself(kind, P):
    """The original project's simple_knn.cu on the same cloud, at a fixed sample of points (tests/golden/make_golden_knn.py)."""
    g = np.load(GOLDEN)
    rows, ref = g["%s_%d_rows" % (kind, P)], g["%s_%d_dist2" % (kind, P)]
    p = _cloud(kind, P)
    np.testing.assert_allclose(_ours(p)[rows], ref, rtol=RTOL, atol=1e-30)
    np.testing.assert_allclose(ref, knn_oracle.dist2_f64(p)[rows], rtol=RTOL, atol=1e-30)       # and the oracle is pinned by it


def test_small_sets_and_empty_input():
    from simple_knn._C import distCUDA2
    p = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [5, 5, 5]], np.float32)
    with np.errstate(over="ignore"):
        for n in (1, 2, 3, 4, 5):
            got, want = _ours(p[:n]), knn_oracle.dist2_f32(p[:n])
            assert np.array_equal(got, want), (n, got, want)
    assert distCUDA2(torch.zeros((0, 3), device="cuda")).shape == (0,)
    with pytest.raises(RuntimeError, match="no CPU path"):
        distCUDA2(torch.zeros((4, 3)))


def test_million_points_against_kdtree_and_stream_order():
    """Size-independent check at 1M points (exact kd-tree) and that the call is stream-ordered (no default-stream use)."""
    from scipy.spatial import cKDTree
    from simple_knn._C import distCUDA2
    p = _cloud("ball", 1_000_000, seed=9)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t = torch.tensor(p, device="cuda")
        got = distCUDA2(t)
    s.synchronize()
    d, _ = cKDTree(p.astype(np.float64)).query(p.astype(np.float64), k=4, workers=-1)
    np.testing.assert_allclose(got.cpu().numpy(), (d[:, 1:] ** 2).mean(axis=1), rtol=RTOL, atol=1e-30)
