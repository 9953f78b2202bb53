"""The flat traversal (scenes of <= 32 leaves: octant-ordered leaf boxes, nearest candidate leaf first, shared exact-test
rounds) against the CPU oracle and against the tree walk, bit for bit.

The ray batch is built to sit on the decisions the box pass and the nearest-leaf step make: axis-parallel directions and
directions with +-0.0 components (inv = +-1e30, the sign of zero picks the octant), origins spawned off every face, rays aimed at
quad diagonals and at the edges and corners two leaves share (equal t in two leaves), NEE-like maxt just short of the target,
and maxt = inf; every direction octant is present."""
import numpy as np
import pytest

from conftest import cbox, materials_cbox

import mitsuba3_b200 as mb
from mitsuba3_b200.integrators import DeviceScene, PathIntegrator

pytestmark = pytest.mark.gpu


def _triangles(sc):
    return np.concatenate([s.vertices[s.faces[:, :3].astype(np.int64), :3] for s in sc.shapes]).astype(np.float64)


def adversarial_rays(sc, seed=0):
    rng = np.random.default_rng(seed)
    tri = _triangles(sc)                                              # (F, 3, 3) world space
    nrm = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    # targets: vertices (corners shared by leaves), edge midpoints (quad diagonals, edges shared by leaves), centroids
    targets = np.concatenate([tri.reshape(-1, 3), 0.5 * (tri + np.roll(tri, 1, axis=1)).reshape(-1, 3), tri.mean(axis=1)])
    targets = np.unique(targets.astype(np.float32), axis=0).astype(np.float64)
    # origins: points on every face, spawned off it along +-n, plus points inside the room
    bary = rng.dirichlet(np.ones(3), size=(tri.shape[0], 6))
    on = np.einsum("fkj,fjc->fkc", bary, tri)
    off = rng.choice([1e-4, 1e-3, 0.05], size=on.shape[:2])[..., None] * rng.choice([-1.0, 1.0], size=on.shape[:2])[..., None]
    origins = np.concatenate([(on + off * nrm[:, None]).reshape(-1, 3), rng.uniform(-0.95, 0.95, size=(256, 3))])
    rays = []
    # 1. origin -> target; maxt = inf, the exact distance, and NEE-like just short of it
    oi = rng.integers(0, len(origins), 60_000); ti = rng.integers(0, len(targets), 60_000)
    o, dv = origins[oi], targets[ti] - origins[oi]
    dist = np.linalg.norm(dv, axis=1)
    keep = dist > 1e-6
    o, dv, dist = o[keep], dv[keep] / dist[keep, None], dist[keep]
    maxt = np.choose(rng.integers(0, 3, len(o)), [np.full(len(o), np.inf), dist, dist * (1 - 1e-3)])
    rays.append(np.concatenate([o, dv, maxt[:, None]], axis=1))
    # 2. axis-parallel directions and directions with +-0.0 components, from every origin
    axis = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], np.float64)
    for a in axis:
        for zero_sign in (1.0, -1.0):
            d = np.where(a == 0, zero_sign * 0.0, a)
            rays.append(np.concatenate([origins, np.tile(d, (len(origins), 1)), np.full((len(origins), 1), np.inf)], axis=1))
    d = rng.normal(size=(len(origins), 3)); d[:, rng.integers(0, 3)] = -0.0
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays.append(np.concatenate([origins, d, np.full((len(origins), 1), 3.4e38)], axis=1))
    # 3. every octant by construction: random directions with forced signs, from origins on the faces
    for oc in range(8):
        d = np.abs(rng.normal(size=(4096, 3))) * np.array([-1.0 if oc >> k & 1 else 1.0 for k in range(3)])
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        o = origins[rng.integers(0, len(origins), 4096)]
        rays.append(np.concatenate([o, d, rng.choice([np.inf, 0.05, 0.5], size=(4096, 1))], axis=1))
    r = np.concatenate(rays).astype(np.float32)
    signs = np.signbit(r[:, 3:6]).astype(int) @ np.array([1, 2, 4])
    assert set(signs.tolist()) == set(range(8))
    return r


@pytest.fixture(scope="module")
def oracle_mod(built):
    from oracle import oracle
    return oracle


@pytest.mark.parametrize("make", [cbox, materials_cbox], ids=["cbox", "materials"])
def test_adversarial_rays_match_oracle_bit_for_bit(make, oracle_mod):
    sc = mb.load_dict(make())
    assert sc.n_triangles <= 256
    ds, orc = DeviceScene(sc), oracle_mod.OracleScene(sc)
    rays = adversarial_rays(sc)
    t, uv, prim, shape = ds.ray_intersect(rays)
    to, uvo, primo, shapeo = orc.ray_intersect(rays)
    assert np.array_equal(shape, shapeo) and np.array_equal(prim, primo)
    hit = shape >= 0
    assert hit.mean() > 0.5
    assert np.array_equal(t[hit].view(np.uint32), to[hit].view(np.uint32))
    assert np.array_equal(uv[hit].view(np.uint32), uvo[hit].view(np.uint32))
    assert np.array_equal(ds.ray_test(rays), orc.ray_test(rays))


@pytest.mark.parametrize("hide_emitters", [False, True])
def test_flat_render_equals_tree_walk_render(hide_emitters, monkeypatch, built):
    """Box filter: the film is written without atomics, so two traversals that find the same hits give the same bits."""
    integ = PathIntegrator(max_depth=8, hide_emitters=hide_emitters)
    flat = mb.load_dict(cbox(res=128, spp=32))
    img_flat = integ.render(flat, spp=32, seed=3)
    monkeypatch.setenv("B200PT_FLAT_TRAVERSAL", "0")             # read when the device scene is created
    walk = mb.load_dict(cbox(res=128, spp=32))
    img_walk = integ.render(walk, spp=32, seed=3)
    assert img_flat.mean() > 0
    assert np.array_equal(img_flat, img_walk)
