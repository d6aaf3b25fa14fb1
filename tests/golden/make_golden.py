#!/usr/bin/env python3
"""Extract the golden vectors the reference ships for the MSM/NTT hot path into small fixtures.

    python tests/golden/make_golden.py <proof-systems checkout>/srs

Run once against a checkout of the reference; the outputs are committed so that the tests need no such checkout.  Apart
from the generator selectors it computes nothing: it only re-packs bytes that the reference's own test
`heavy_test_srs_serialization` (poly-commitment/src/precomputed_srs.rs:156-234) asserts equal to a fresh SRS::create + get_lagrange_basis.

Sources (formats: SURVEY.md Appendix B, poly-commitment/src/precomputed_srs.rs:38-51,
utils/src/serialization.rs:65-146):
  srs/pallas.srs, srs/vesta.srs            [g (65536 x 33 B compressed), h]
  srs/test_pallas.srs, srs/test_vesta.srs  [g (65 B uncompressed), h, {n: [[point]]} Lagrange bases n = 1..65536]

Outputs (tests/golden/):
  pallas_srs.npz  g_sel      uint8 [65536]     how to rebuild compressed g (all of it: config 2 needs the 2^16-point SRS),
                                               see tests/golden/srs_fixture.py
                  g_cmp_sha256 uint8 [32]      sha256 of the reference's compressed g (65536 x 33 bytes)
                  g_xy       uint8 [2048,64]   canonical LE x||y of g[0..2048] (cross-pins decompression)
                  h_xy       uint8 [64]
                  lag_2048   uint8 [2048,64]   lagrange_bases[2048][i] for all i  (config 1: 2048 pinned 2^11-point MSMs)
                  lag_small  uint8 [2047,64]   lagrange_bases[n][i], n = 1,2,..,1024 concatenated
                  lag_65536_idx int64 [k], lag_65536 uint8 [k,64]   sampled answers of 2^16-point MSMs
                  lag_65536_sha256 uint8 [32]   sha256 of the whole stored 2^16 basis (65536 x 64 canonical bytes, index order)
  vesta_srs.npz   the same keys
"""
import os
import sys

import msgpack
import numpy as np

import srs_fixture

OUT = os.path.dirname(os.path.abspath(__file__))
SAMPLE_65536 = [0, 1, 2, 3, 1000, 32768, 40000, 65534, 65535]


def load(path):
    with open(path, "rb") as f:
        return msgpack.unpackb(f.read(), strict_map_key=False)


def xy(b: bytes) -> np.ndarray:
    assert len(b) == 65 and b[64] == 0, "expected finite uncompressed point"
    return np.frombuffer(b[:64], dtype=np.uint8)


def selectors(curve, g_cmp):
    """g_sel of srs_fixture: which candidate x of the map is g[i]'s (checked to be the first with a square x^3 + 5), y flag"""
    sel = np.empty(len(g_cmp), dtype=np.uint8)
    for i, p in enumerate(g_cmp):
        x = int.from_bytes(p[:32].tobytes(), "little")
        xs = srs_fixture.candidate_xs(curve, srs_fixture.map_input(i))
        k = next(k for k, c in enumerate(xs) if srs_fixture.is_square(curve, c))
        assert xs[k] == x and p[32] in (0, 0x80), f"{curve} g[{i}] is not the map's point"
        sel[i] = k | p[32]
    return sel


def main(ref):
    for curve in ("pallas", "vesta"):
        small = load(os.path.join(ref, f"{curve}.srs"))
        test = load(os.path.join(ref, f"test_{curve}.srs"))
        g_c, h_c = small
        g_u, h_u, lag = test
        assert len(g_c) == 65536 and len(g_u) == 65536
        keep = 65536          # both curves keep every generator since round 2: the 2^16 prover replay (tests/test_gpu_replay.py) commits on Vesta
        g_cmp = np.stack([np.frombuffer(p, dtype=np.uint8) for p in g_c[:keep]])
        g_xy = np.stack([xy(p) for p in g_u[:2048]])
        # the two files agree on x for every generator
        for i in range(65536):
            assert g_c[i][:32] == g_u[i][:32]
        lag_2048 = np.stack([xy(c[0]) for c in lag[2048]])
        lag_small = np.concatenate([np.stack([xy(c[0]) for c in lag[1 << k]]) for k in range(11)])
        assert lag_small.shape == (2047, 64)
        lag_65536 = np.stack([xy(lag[65536][i][0]) for i in SAMPLE_65536])
        # the WHOLE stored 2^16 basis, pinned by digest: 65536 x (x || y), canonical LE, in index order
        import hashlib
        digest = hashlib.sha256(b"".join(bytes(lag[65536][i][0][:64]) for i in range(65536))).digest()
        g_sel = selectors(curve, g_cmp)
        assert np.array_equal(srs_fixture.generators(curve, g_sel), g_cmp)
        np.savez_compressed(
            os.path.join(OUT, f"{curve}_srs.npz"),
            g_sel=g_sel,
            g_cmp_sha256=np.frombuffer(hashlib.sha256(g_cmp.tobytes()).digest(), dtype=np.uint8),
            g_xy=g_xy,
            h_xy=xy(h_u),
            lag_2048=lag_2048,
            lag_small=lag_small,
            lag_65536_idx=np.array(SAMPLE_65536, dtype=np.int64),
            lag_65536=lag_65536,
            lag_65536_sha256=np.frombuffer(digest, dtype=np.uint8),
        )
        print(curve, "ok", os.path.getsize(os.path.join(OUT, f"{curve}_srs.npz")))


if __name__ == "__main__":
    sys.exit(main(sys.argv[1]))
