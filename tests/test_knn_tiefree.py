"""The k-best insertion compares dis2 alone and looks original indices up only for the slots whose dis2 a candidate
ties (knn_insert / knn_seed, voxel_map.cuh).  These maps are built so that exact float32 distance ties are the rule:
dyadic lattice coordinates (every dis2 exact), queries on and between lattice points (points symmetric about the
query), and repeated coordinates under distinct indices (masked duplicates, quirk Q3).  Every search form - unseeded,
seeded with tied seeds, tracked (the K-set re-sort) - must return the exact (dis2, original index) order.  d6 is not
read out: it is checked only through the tracked results, which a margin that came out too large would make wrong."""
import numpy as np
import pytest

import hostsim_py as HS
import oracle_py as O


def _lattice(n_side, step, layers, seed):
    g = (np.arange(n_side, dtype=np.float32) - np.float32(n_side // 2)) * np.float32(step)
    x, y, z = np.meshgrid(g, g, g[:layers])
    pts = np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float32)
    rng = np.random.default_rng(seed)
    return pts[rng.permutation(len(pts))]


def _cloud(pts):
    return np.concatenate([pts, np.zeros((len(pts), 1), np.float32)], 1)


def _queries(pts, step, seed):
    rng = np.random.default_rng(seed)
    base = pts[rng.choice(len(pts), 600, replace=False)]
    # on a lattice point, half a step off along one, two or three axes: all of them sit on symmetry planes of the lattice
    offs = np.array([[0, 0, 0], [0.5, 0, 0], [0.5, 0.5, 0], [0.5, 0.5, 0.5], [0.25, 0, 0], [0.25, 0.25, 0.5]], np.float32)
    return (base + offs[np.arange(len(base)) % len(offs)] * np.float32(step)).astype(np.float32)


@pytest.fixture(scope="module", params=[(0.25, 0.5), (0.125, 0.5), (0.5, 0.3)], ids=["dense", "denser", "sparse"])
def tied(request):
    step, cell = request.param
    pts = _lattice(24, step, 5, seed=1)
    # every 7th point again under a new index: same coordinates, only the lowest index may be returned
    pts = np.concatenate([pts, pts[::7]])
    pts = pts[np.random.default_rng(2).permutation(len(pts))]
    cloud = _cloud(pts)
    ref = O.OracleIcp(method=O.P2PLANE, nn_mode=O.NN_EXACT_TIEBREAK, skip_nonfinite=1)  # de-duplicates as the map does
    ref.set_target(cloud)
    return ref, HS.HsMap(cloud, cell=cell), _queries(pts, step, seed=3), step


def test_unseeded_search_with_ties(tied):
    ref, m, q, _ = tied
    for k in (1, 5):
        assert np.array_equal(m.knn(q, k), ref.knn(q, k))


def test_seeded_search_with_tied_seeds(tied):
    """Seeds found at a lattice point of their own: their five distances tie in pairs at the query (the sorting network's
    index fallback), and the list scan meets them again."""
    ref, m, q, step = tied
    exp = ref.knn(q, 5)
    for shift in ((0, 0, 0), (step, 0, 0), (0.5 * step, 0.5 * step, 0), (0, 0, 2 * step)):
        assert np.array_equal(m.knn_seeded(q, (q + np.float32(shift)).astype(np.float32)), exp), shift


@pytest.mark.parametrize("k", [1, 5])
def test_tracked_search_with_ties(tied, k):
    """The tracked form (the K-set shortcut and the margins it relies on) over steps that stay on the symmetry planes: a tie at the
    K-th leaves no margin, so these queries search every time; steps off the planes may take the shortcut."""
    ref, m, q, step = tied
    rng = np.random.default_rng(4)
    moves = [0.0, 0.0, 0.5 * step, 1e-4, 0.0, 0.25 * step, 1e-5, 0.0]
    steps = np.stack([(q + np.float32(d) * rng.integers(-1, 2, q.shape).astype(np.float32)).astype(np.float32) for d in moves])
    got, _ = m.knn_tracked(steps, k)
    for s in range(len(moves)):
        assert np.array_equal(got[s], ref.knn(steps[s], k)), s
