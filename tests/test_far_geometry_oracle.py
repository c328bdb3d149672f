"""CPU suite: the oracle's BVH against its own brute force (every ray against every triangle) on scenes far from the origin,
scaled, and seeded with ties.  The BVH's box padding has to survive coordinate rounding: once ulp(max |coord|) exceeds the
1e-4 x extent padding, a ray lying in a box's face plane reads 0 * inf there and the slab test drops the box that holds
its hit.  The GPU tests use the brute force as their reference; this keeps the oracle's BVH honest without a GPU."""
import numpy as np
import pytest

import geometry_scenes as gs
from oracle.pyoracle import Oracle

CORNELL_KEYS = list(gs.OFFSETS) + list(gs.SCALES)


def _same_hits(a, b):
    return (np.array_equal(a["triangleId"], b["triangleId"]) and np.array_equal(a["t"].view(np.uint32), b["t"].view(np.uint32))
            and np.array_equal(a["u"].view(np.uint32), b["u"].view(np.uint32)) and np.array_equal(a["v"].view(np.uint32), b["v"].view(np.uint32)))


@pytest.mark.parametrize("key", CORNELL_KEYS)
def test_oracle_bvh_equals_brute_cornell(key, uv50):
    sc = gs.with_ties(gs.cornell512_at(key))
    orc = Oracle.from_scene(sc)
    pair = np.concatenate([orc.pair_rays(i, j, uv50) for i, j in [(0, 511), (3, 100), (17, 300), (40, 41), (200, 450)]])
    rays = np.concatenate([gs.closest_hit_rays(sc, 1), pair])
    want = orc.query_closest(rays, brute=True)
    assert (want["triangleId"] >= 0).mean() > 0.8
    assert _same_hits(orc.query_closest(rays), want), key


@pytest.mark.parametrize("name", ["irregular1", "irregular2", "perforated1", "perforated2"])
def test_oracle_bvh_equals_brute_walls_far(name):
    base = gs.irregular_walls(int(name[-1])) if name.startswith("irregular") else gs.perforated_plate(int(name[-1]))
    sc = gs.moved(base, offset=gs.FAR_DIRECTION_32768)
    orc = Oracle.from_scene(sc)
    rays = gs.closest_hit_rays(sc, 2)
    want = orc.query_closest(rays, brute=True)
    assert (want["triangleId"] >= 0).mean() > 0.3
    assert _same_hits(orc.query_closest(rays), want), name


@pytest.mark.parametrize("key", ["o16384", "o32768", "o3e5"])
def test_oracle_bvh_equals_brute_form_factor_rows(key, uv50):
    """Masks and matrix rows of the BVH-accelerated build against the brute-force build of the same translated scene."""
    sc = gs.cornell512_at(key)
    orc = Oracle.from_scene(sc)
    rows = np.arange(0, 512, 9)
    F, m, _ = orc.radmat_rowlist(uv50, rows)
    F_ref, m_ref, _ = orc.radmat_rowlist(uv50, rows, brute=True)
    assert (m_ref != 0).sum() > 1000
    assert np.array_equal(m, m_ref)
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
