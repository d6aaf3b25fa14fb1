"""pytest configuration: the `gpu` marker and shared fixtures (golden SRS vectors, oracle handle)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
if GOLDEN not in sys.path:
    sys.path.insert(0, GOLDEN)
import srs_fixture  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def orc():
    from oracle import oracle
    oracle.lib()
    return oracle


class GoldenSRS:
    """Golden vectors of one curve (see tests/golden/make_golden.py), decoded to the library's conventions."""

    def __init__(self, curve_name, orc):
        self.cid = orc.PALLAS if curve_name == "pallas" else orc.VESTA
        self.base = orc.BASE_FIELD[self.cid]
        self.scalar = orc.SCALAR_FIELD[self.cid]
        z = srs_fixture.load(curve_name)
        self.g_cmp = z["g_cmp"]                      # uint8 [k,33]
        self.g_xy_canon = z["g_xy"]                  # uint8 [2048,64]
        self.h_xy_canon = z["h_xy"]
        self.lag_2048_canon = z["lag_2048"]
        self.lag_small_canon = z["lag_small"]
        self.lag_65536_idx = z["lag_65536_idx"]
        self.lag_65536_canon = z["lag_65536"]
        self._orc = orc
        self._g = None

    def mont_points(self, canon_u8):
        """uint8 [...,64] canonical LE x||y -> uint64 [...,8] Montgomery affine"""
        a = np.ascontiguousarray(canon_u8).view("<u8").reshape(-1, 4)
        return self._orc.to_mont(self.base, a).reshape(-1, 8)

    @property
    def g(self):
        """All generators kept in the fixture, decompressed by the oracle: uint64 [k,8] Montgomery."""
        if self._g is None:
            self._g = self._orc.decompress(self.cid, self.g_cmp.tobytes())
        return self._g

    def lagrange_small(self, n):
        """lagrange_bases[n] for n in {1,2,...,1024}: uint64 [n,8] Montgomery"""
        off = n - 1
        return self.mont_points(self.lag_small_canon[off:off + n])


@pytest.fixture(scope="session")
def pallas_srs(orc):
    return GoldenSRS("pallas", orc)


@pytest.fixture(scope="session")
def vesta_srs(orc):
    return GoldenSRS("vesta", orc)
