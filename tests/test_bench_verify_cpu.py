"""CPU checks of bench.py's self-verification helpers (closed form of SURVEY.md §8(c) L1, Horner evaluation) against the
big-int oracle, and of the five BASELINE schedules (MSM counts of the SURVEY.md §8 table)."""
import numpy as np
import bench
from oracle import pyref
from util import mont, rand_ints, affine_to_limbs, ints_to_limbs


def test_schedule_counts_match_survey_table():
    want = {1: (14, 8), 2: (16, 28), 3: (19, 12), 4: (20, 32), 5: (23, 12)}
    for cid, (k, msms) in want.items():
        s = bench.Schedule(cid)
        assert (s.k, len(s.msm)) == (k, msms)
        assert sum(len(p) for p in s.phases) == msms
        assert sorted(i for v in s.ntt_ready.values() for i in v) == list(range(s.n_poly))
    assert bench.Schedule(3).ext_k == 21 and bench.Schedule(1).ext_k == 15 and bench.Schedule(4).ext_k == 22


def test_progression_dot_and_point_match():
    rng = np.random.default_rng(5)
    n, begin, a0, d = 300, 40, 7, 11
    s = rand_ints(rng, n, pyref.R)
    m = mont(s, pyref.R)
    dot = bench.progression_dot(m, a0, d, begin)
    want = sum(pyref.to_mont(si, pyref.R) * (a0 + d * (begin + i)) for i, si in enumerate(s))
    assert dot == want
    scalar = dot * bench.MONT_RINV_R % bench.R_MOD
    assert scalar == sum(si * (a0 + d * (begin + i)) for i, si in enumerate(s)) % pyref.R
    pt = bench.ec_mul_g(scalar)
    assert pt == pyref.g1_mul(scalar, pyref.G1)
    # a Jacobian representative with z != 1, Montgomery limbs, as the library returns it
    z = 0x1234567
    X, Y = pt[0] * z * z % pyref.P, pt[1] * z * z * z % pyref.P
    limbs = ints_to_limbs([pyref.to_mont(v, pyref.P) for v in (X, Y, z)]).reshape(12)
    assert bench.point_matches(limbs, pt)
    bad = limbs.copy(); bad[0] ^= np.uint64(1)
    assert not bench.point_matches(bad, pt)
    ident = ints_to_limbs([0, pyref.to_mont(1, pyref.P), 0]).reshape(12)
    assert bench.point_matches(ident, None) and not bench.point_matches(ident, pt)
    assert bench.ec_mul_g(0) is None and bench.ec_mul_g(pyref.R) is None and bench.ec_mul_g(1) == (1, 2)


def test_horner_mont():
    rng = np.random.default_rng(6)
    c = rand_ints(rng, 50, pyref.R)
    x = 0xabcdef123
    assert bench.horner_mont(mont(c, pyref.R), x) == sum(ci * pow(x, i, pyref.R) for i, ci in enumerate(c)) % pyref.R
    assert bench.ZETA == pyref.ZETA and bench.ROOT_OF_UNITY == pyref.ROOT_OF_UNITY


def test_dump_outputs_are_canonical_values():
    """--dump-outputs writes values, not representations: Montgomery limbs and Jacobian points come out as the integers
    they stand for, in exact 32-bit limbs; the sampled rows are fixed and every schedule's dump fits the size limit"""
    rng = np.random.default_rng(7)
    s = rand_ints(rng, 20, pyref.R) + [0, 1, pyref.R - 1]
    got = bench.fr_canonical(mont(s, pyref.R))
    assert got.dtype == np.float64 and got.shape == (len(s), 8)
    assert [sum(int(l) << (32 * i) for i, l in enumerate(row)) for row in got] == s
    pt = pyref.g1_mul(0xfeed, pyref.G1)
    z = 0x7654321
    jac = ints_to_limbs([pyref.to_mont(v, pyref.P) for v in (pt[0] * z * z % pyref.P, pt[1] * z ** 3 % pyref.P, z)]).reshape(12)
    aff = bench.g1_affine(jac)
    assert [sum(int(l) << (32 * i) for i, l in enumerate(aff[h:h + 8])) for h in (0, 8)] == list(pt)
    assert not bench.g1_affine(ints_to_limbs([0, pyref.to_mont(1, pyref.P), 0]).reshape(12)).any()
    rows = bench.dump_rows(1 << 21)
    assert len(rows) == bench.DUMP_ROWS and np.array_equal(rows, bench.dump_rows(1 << 21)) and np.all(np.diff(rows) > 0)
    assert np.array_equal(bench.dump_rows(100), np.arange(100))
    for cfg in (1, 2, 3, 4, 5):
        sc = bench.Schedule(cfg)
        arrays = sc.A + sc.L + 2 * sc.n_poly  # assigned columns, coefficients, extended + extended_to_coeff
        assert len(sc.msm) * 16 * 8 + arrays * bench.DUMP_ROWS * 8 * 8 <= bench.DUMP_LIMIT


def test_every_transform_has_one_owner_at_every_world_size():
    """bench.py deals whole transforms to the ranks by cost; at 8 GPUs some ranks own only a coset transform or none at
    all (the k = 14 config has 7 transforms) — every transform must still have exactly one owner"""
    import bench
    import halo2_lib_b200 as h
    for cfg in (1, 2, 3, 4, 5):
        s = bench.Schedule(cfg)
        costs = [1.0] * s.n_poly + [float(1 << (s.ext_k - s.k))] * (s.n_poly + 1)
        for world in (1, 2, 4, 8):
            owners = h.ntt_owners_balanced(costs, world)
            assert len(owners) == 2 * s.n_poly + 1 and all(0 <= o < world for o in owners)
            load = [sum(c for c, o in zip(costs, owners) if o == r) for r in range(world)]
            assert max(load) - min(load) <= max(costs)
