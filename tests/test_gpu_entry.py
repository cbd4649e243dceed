"""Every pair call on one device checks every set id it names before it computes anything, also when it has no pairs:
an id past the last set is GKD_EINVAL and a set that has not been built is GKD_ESTATE, whatever the form and however
many pairs the call has."""
import numpy as np
import pytest

import genome.distance_b200 as gkd

pytestmark = pytest.mark.gpu

EINVAL, ESTATE = -1, -5


def _code(call):
    with pytest.raises(gkd.GkdError) as err:
        call()
    return err.value.code


def test_triangle_of_one_unbuilt_set():
    with gkd.Engine(k=21) as e:
        e.add("ACGT" * 100)
        assert _code(lambda: e.all_vs_all()) == ESTATE
        assert _code(lambda: e.all_vs_all_linkage(0.5)) == ESTATE
        e.build()
        a, b, inter, dist = e.all_vs_all_linkage(0.5)
        assert a.size == b.size == inter.size == dist.size == 0


def test_rectangle_with_an_empty_side_checks_the_other_side():
    rng = np.random.default_rng(11)
    with gkd.Engine(k=21) as e:
        for _ in range(2):
            e.add(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), 4000).tobytes().decode())
        e.build()
        e.add("ACGT" * 100)  # set 2, never built
        forms = {
            "dense": lambda q, r: e.query_vs_ref(q, r),
            "within": lambda q, r: e.query_vs_ref_within(q, r, 0.5),
            "nearest": lambda q, r: e.query_vs_ref_nearest(q, r, 3, 1.0),
            "nearest_ex": lambda q, r: e.query_vs_ref_nearest_ex(q, r, 3, 1.0),
            "clusters": lambda q, r: e.query_vs_ref_clusters(q, r, 0.5),
            "linkage": lambda q, r: e.query_vs_ref_linkage(q, r, 0.5),
        }
        for name, call in forms.items():
            for bad, code in ((999, EINVAL), (2, ESTATE)):
                assert _code(lambda: call([bad], [])) == code, (name, bad)
                assert _code(lambda: call([], [bad])) == code, (name, bad)
            # the same calls over built sets answer
            call([1], [])
            call([], [1])
