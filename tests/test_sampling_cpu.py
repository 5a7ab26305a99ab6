"""CPU: the numpy restatement of the library's random streams (philox_ref.py) and the counters the GPU sampling tests
hard-code."""
import numpy as np
import pytest

import philox_ref as P
from test_gpu_sampling import CASES, EDGE_DRAWS


def _words(c):
    return " ".join("%08x" % int(v) for v in c)


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, want):
    """Random123's known-answer vectors for Philox4x32-10."""
    assert _words(P.philox4x32_10(ctr, key)) == want


def test_philox_vectorised_equals_scalar():
    ctr = np.arange(64, dtype=np.uint64) * np.uint64(0x01000193)
    got = P.philox4x32_10((ctr, ctr + np.uint64(1), ctr >> np.uint64(3), 7), (0x12345678, ctr))
    for i in (0, 17, 63):
        one = P.philox4x32_10((int(ctr[i]), int(ctr[i]) + 1, int(ctr[i]) >> 3, 7), (0x12345678, int(ctr[i])))
        assert [int(w[i]) for w in got] == [int(w) for w in one]


def test_uniform_mapping_end_points():
    """((x >> 8) + 0.5f) * 2^-24: x >> 8 = 0 gives 2^-25; 2^24 - 1 + 0.5 rounds to 2^24 in fp32 (ties to even), so the
    largest value is exactly 1.0 and the draw must be able to reach the end of the CDF."""
    top = np.uint64(0xFFFFFF00)
    assert P.uniform_from_word(np.uint64(0)) == np.float32(2.0 ** -25) == P.U_BOTTOM
    assert P.uniform_from_word(np.uint64(0xFF)) == P.U_BOTTOM
    assert P.uniform_from_word(top) == np.float32(1.0) == P.U_TOP
    assert P.uniform_from_word(top - np.uint64(0x100)) < 1.0
    assert P.uniform_from_word(top).dtype == np.float32
    k = np.arange(2 ** 24 - 16, 2 ** 24, dtype=np.uint64) << np.uint64(8)
    u = P.uniform_from_word(k)
    assert np.all(np.diff(u) >= 0) and np.all(u <= 1.0)


def test_sample_uniform_counter_layout():
    """grow fills counter words 0-1, step words 2-3, seed the key: every word changes the draw, and the 64-bit halves
    are not folded together."""
    base = P.sample_uniform(5, 7, 3)
    assert base == P.uniform_from_word(P.philox4x32_10((7, 0, 3, 0), (5, 0))[0])
    assert P.sample_uniform(5 + 2 ** 32, 7 + 2 ** 32, 3 + 2 ** 32) == \
        P.uniform_from_word(P.philox4x32_10((7, 1, 3, 1), (5, 1))[0])
    others = [P.sample_uniform(5, 8, 3), P.sample_uniform(5, 7, 4), P.sample_uniform(6, 7, 3),
              P.sample_uniform(5, 7 + 2 ** 32, 3), P.sample_uniform(5, 7, 3 + 2 ** 32), P.sample_uniform(5 + 2 ** 32, 7, 3)]
    assert all(o != base for o in others)
    rows = P.sample_uniform(5, np.arange(1000, dtype=np.uint64), 3)
    assert rows.shape == (1000,) and len(np.unique(rows)) == 1000
    assert abs(float(rows.mean()) - 0.5) < 0.05


def test_hard_coded_edge_counters_hit_the_ends():
    """The (seed, row, step) triples of test_gpu_sampling really map to the smallest and largest uniform."""
    for _, step, seed, grow, want in EDGE_DRAWS:
        assert P.sample_uniform(seed, grow, step) == want, (seed, grow, step)
    tops = [e for e in EDGE_DRAWS if e[4] == P.U_TOP]
    bottoms = [e for e in EDGE_DRAWS if e[4] == P.U_BOTTOM]
    n_rollout = 0
    for c in CASES:
        for b, m, t in c["edges"]:
            assert P.sample_uniform(c["seed"], b * c["M"] + m, t) == P.U_TOP, c["id"]
            assert t >= (2 if c["kind"] == "cvrp" else 1) and t < c["N"] - 1 and b < c["n"] * c["aug"] and m < c["M"]
            n_rollout += 1
    assert len(tops) + n_rollout >= 16 and len(bottoms) >= 2 and n_rollout >= 1


def test_generator_restatement_shapes_and_exact_parts():
    """The restated generator on the CPU alone: exact uniform coordinates, integer demands, the depot split of cvrp
    cluster, the mutated half of mixed."""
    u = P.generate("cvrp", 0, 3, 20, 1, 0.2, 0.8, 0.07, 30.0, seed=9)
    assert u["node"].shape == (3, 20, 2) and u["depot"].shape == (3, 2) and not u["gauss"].any()
    assert np.all((u["node"] >= 0) & (u["node"] < 1)) and np.all(u["node"] * 2 ** 24 == np.round(u["node"] * 2 ** 24))
    q = u["demand"] * np.float32(30.0)
    assert np.all(np.abs(q - np.round(q)) < 1e-5) and q.min() >= 1 and q.max() <= 9
    c = P.generate("cvrp", 1, 2, 21, 3, 0.2, 0.8, 0.07, 30.0, seed=9)
    assert np.all((c["depot_idx"] >= 0) & (c["depot_idx"] <= 21)) and c["gauss"].all() and c["depot_gauss"].all()
    m = P.generate("tsp", 2, 2, 21, 1, 0.2, 0.8, 0.07, 1.0, seed=9)
    assert (m["mutated"].sum(1) == 10).all() and np.array_equal(m["gauss"], m["mutated"])
    assert np.array_equal(P.generate("tsp", 2, 2, 21, 1, 0.2, 0.8, 0.07, 1.0, seed=9)["node"], m["node"])
