"""The MSM launch chain (option msm_pdl): kernels after the first launched by programmatic dependent launch, empty buckets set by
the plan kernel and the histogram counted back to zero by the scatter instead of two memsets per call.  The earlier launch shell
(plain launches behind the memsets, msm_pdl = 0) must return the same affine points on the same inputs, and switching between
the two on one workspace must leave it clean."""
import numpy as np
import pytest

import proof_systems_b200 as zk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = zk.Context(0)
    yield c
    c.close()


def both(ctx, curve, fn):
    """fn() under the PDL chain and under the plain launch shell, new first then old then new again; affine results"""
    out = []
    try:
        for pdl in (1, 0, 1):
            ctx.set_option("msm_pdl", pdl)
            out.append(zk.jacobian_to_affine(curve, fn()))
    finally:
        ctx.set_option("msm_pdl", 1)
    assert np.array_equal(out[0], out[1]) and np.array_equal(out[0], out[2])
    return out[0]


def test_headline_2_16_window_16(ctx, orc, pallas_srs):
    srs = pallas_srs
    n = 1 << 16
    sc = orc.random_scalars(srs.scalar, n, seed=21)
    bases = ctx.upload_bases(srs.cid, srs.g[:n], window_bits=16)
    both(ctx, srs.cid, lambda: ctx.msm(bases, sc))
    bases.free()


@pytest.mark.parametrize("kind", ["random", "zeros", "ones", "sparse16"])
def test_2_11_default_window(ctx, orc, pallas_srs, kind):
    """random scalars; all zero (every bucket empty: the identity); all one (one giant bucket); 5 % non-zero 16-bit scalars
    (most buckets empty)"""
    srs = pallas_srs
    n = 1 << 11
    if kind == "random":
        sc = orc.random_scalars(srs.scalar, n, seed=22)
    elif kind == "zeros":
        sc = np.zeros((n, 4), dtype=np.uint64)
    elif kind == "ones":
        sc = np.zeros((n, 4), dtype=np.uint64)
        sc[:, 0] = 1
    else:
        sc = orc.random_scalars(srs.scalar, n, seed=23)
        sc[:, 1:] = 0
        sc[:, 0] &= 0xffff
        sc[np.random.default_rng(5).random(n) >= 0.05] = 0
    bases = ctx.upload_bases(srs.cid, srs.g[:n], window_bits=-1)
    got = both(ctx, srs.cid, lambda: ctx.msm(bases, sc))
    assert np.array_equal(got, orc.msm(srs.cid, srs.g[:n], sc))
    bases.free()


def test_batch_of_15_with_offset(ctx, orc, vesta_srs):
    srs = vesta_srs
    n, k, off = 1500, 15, 300
    bases = ctx.upload_bases(srs.cid, srs.g[:2048], window_bits=-1)
    sc = orc.random_scalars(srs.scalar, n * k, seed=24).reshape(k, n, 4)
    out = []
    try:
        for pdl in (1, 0):
            ctx.set_option("msm_pdl", pdl)
            out.append(ctx.msm_batch(bases, sc, off=off))
    finally:
        ctx.set_option("msm_pdl", 1)
    for j in range(k):
        a, b = (zk.jacobian_to_affine(srs.cid, o[j]) for o in out)
        assert np.array_equal(a, b), j
    assert np.array_equal(zk.jacobian_to_affine(srs.cid, out[0][k - 1]), orc.msm(srs.cid, srs.g[off:off + n], sc[k - 1]))
    bases.free()


def test_ipa_rounds_lr(ctx, orc, pallas_srs):
    """the L / R pair of every IPA round: a batch of two MSMs at offsets 0 and n/2 over a shrinking folded base set"""
    srs = pallas_srs
    n = 256
    a = orc.to_mont(srs.scalar, orc.random_scalars(srs.scalar, n, seed=25))
    b = orc.to_mont(srs.scalar, orc.random_scalars(srs.scalar, n, seed=26))
    chals = orc.to_mont(srs.scalar, orc.random_scalars(srs.scalar, 8, seed=27))
    bases = ctx.upload_bases(srs.cid, srs.g[:n], window_bits=-1)
    res = {}
    try:
        for pdl in (1, 0):
            ctx.set_option("msm_pdl", pdl)
            rounds = zk.IpaRounds(ctx, bases, a, b)
            seq = []
            for u in chals:
                l, r, _, _ = rounds.lr()
                seq.append((zk.jacobian_to_affine(srs.cid, l), zk.jacobian_to_affine(srs.cid, r)))
                rounds.fold(u, u)      # any scalar folds; both paths fold with the same one
            rounds.close()
            res[pdl] = seq
    finally:
        ctx.set_option("msm_pdl", 1)
    for (l1, r1), (l0, r0) in zip(res[1], res[0]):
        assert np.array_equal(l1, l0) and np.array_equal(r1, r0)
    bases.free()


def test_calls_of_different_size_on_one_workspace(orc, vesta_srs):
    """a fresh context: a small call, a call that grows every workspace buffer, a small one again — the histogram must start
    from zero in each, on both launch shells"""
    srs = vesta_srs
    c = zk.Context(0)
    try:
        small = c.upload_bases(srs.cid, srs.g[:2048], window_bits=-1)
        big = c.upload_bases(srs.cid, srs.g, window_bits=-1)
        n_big = len(srs.g)
        s1 = orc.random_scalars(srs.scalar, 2048, seed=28)
        s2 = orc.random_scalars(srs.scalar, n_big, seed=29)
        want1 = orc.msm(srs.cid, srs.g[:2048], s1)
        want2 = orc.msm(srs.cid, srs.g, s2)
        for pdl in (1, 0, 1):
            c.set_option("msm_pdl", pdl)
            assert np.array_equal(c.msm_affine(small, s1), want1), pdl
            assert np.array_equal(c.msm_affine(big, s2), want2), pdl
            assert np.array_equal(c.msm_affine(small, s1[:1000]), orc.msm(srs.cid, srs.g[:1000], s1[:1000])), pdl
        small.free()
        big.free()
    finally:
        c.close()


def test_launch_count_and_option_range(ctx, pallas_srs):
    srs = pallas_srs
    n = 1 << 11
    bases = ctx.upload_bases(srs.cid, srs.g[:n], window_bits=16)
    sc = np.ones((n, 4), dtype=np.uint64)
    counts = []
    try:
        for pdl in (1, 0):
            ctx.set_option("msm_pdl", pdl)
            l0 = ctx.launch_count
            ctx.msm(bases, sc)
            counts.append(ctx.launch_count - l0)
    finally:
        ctx.set_option("msm_pdl", 1)
    assert counts[0] == counts[1] >= 9      # recode, plan, scatter, accumulate, giant finish, run sum, bucket finish, gridsum x2
    with pytest.raises(zk.ZkError):
        ctx.set_option("msm_pdl", 2)
    bases.free()
