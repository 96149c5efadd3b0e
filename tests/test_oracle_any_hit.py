"""tests/any_hit_ref.cpp (the oracle's Occluders::anyHit over a whole triangle list, multithreaded) against the OR of the
oracle's one-triangle entry gvpm_oracle_pin_triangle over every triangle: the reference answer of the occluder any-hit
tests."""
import numpy as np
import pytest

import any_hit_ref as AH
import occluder_sets as S


@pytest.mark.parametrize("which", ["walls", "blocker", "sphere", "soup"])
def test_oracle_any_hit_equals_or_of_single_triangles(which):
    tri = {"walls": S.walls, "blocker": lambda: np.concatenate([S.walls(), S.blocker_sheets()]),
           "sphere": lambda: S.uv_sphere(16, 10), "soup": lambda: S.soup(300, seed=5, size=0.05)}[which]()
    o, d, mint, maxt = S.adversarial_rays(tri, n=4000, seed=13)
    got = AH.any_hit(tri, o, d, mint, maxt, threads=4)
    want = S.oracle_any_hit_by_triangle(tri, o, d, mint, maxt)
    np.testing.assert_array_equal(got, want)
    assert got.any() and not got.all()
    # single-threaded gives the same answer
    np.testing.assert_array_equal(AH.any_hit(tri, o, d, mint, maxt, threads=1), got)
