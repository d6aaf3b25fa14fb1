"""The SRS file codec (proof_systems_b200/srs_file.py) against the reference's on-disk format
(poly-commitment/src/precomputed_srs.rs:38-51,76-91; utils/src/serialization.rs:65-146; SURVEY.md Appendix B).
The writer, fed with the fixture's copy of the generators, must reproduce srs/pallas.srs byte for byte (digest pinned here)."""
import hashlib
import os

import numpy as np
import pytest

from proof_systems_b200 import srs_file

# sha256 of /root/reference/srs/pallas.srs (2 293 801 bytes), taken in the build container by tests/golden/make_golden.py's sources
PALLAS_SRS_SHA256 = "c2e2ec94b00252643077d1a5361612891ec5296871f7d8a2d3addf61d065dc23"


def compress_xy(orc, fid, xy64: np.ndarray) -> np.ndarray:
    """canonical x||y (64 bytes) -> 33-byte ark compressed form, with Python integers"""
    m = orc.FP_MODULUS if fid == orc.FP else orc.FQ_MODULUS
    y = int.from_bytes(bytes(xy64[32:]), "little")
    return np.frombuffer(bytes(xy64[:32]) + bytes([0x80 if y > m - y else 0]), dtype=np.uint8)


def test_writer_reproduces_the_reference_file(orc, pallas_srs, tmp_path):
    h = compress_xy(orc, orc.FP, pallas_srs.h_xy_canon)
    path = str(tmp_path / "pallas.srs")
    srs_file.write_srs(path, srs_file.SrsFile(g=pallas_srs.g_cmp, h=h))
    raw = open(path, "rb").read()
    assert len(raw) == 2293801 and raw[:6] == bytes.fromhex("92dd00010000") and raw[6:8] == bytes.fromhex("c421")
    assert hashlib.sha256(raw).hexdigest() == PALLAS_SRS_SHA256
    back = srs_file.read_srs(path)
    assert back.compressed and np.array_equal(back.g, pallas_srs.g_cmp) and np.array_equal(back.h, h) and not back.lagrange_bases


@pytest.mark.parametrize("name", ["pallas", "vesta"])
def test_rebuilt_generators_are_the_reference_ones(request, name):
    """The fixture's 2^16 generators, rebuilt by tests/golden/srs_fixture.py, are byte for byte those of srs/<name>.srs, and the
    stored selectors agree with the map's rule (the first candidate x whose x^3 + 5 is a square) on a sample."""
    import srs_fixture
    G = request.getfixturevalue(f"{name}_srs")
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"{name}_srs.npz"))
    assert G.g_cmp.shape == (1 << 16, 33)
    assert hashlib.sha256(G.g_cmp.tobytes()).digest() == z["g_cmp_sha256"].tobytes()
    for i in list(range(64)) + [1000, 32768, 65535]:
        xs = srs_fixture.candidate_xs(name, srs_fixture.map_input(i))
        assert int(z["g_sel"][i]) & 3 == next(k for k, x in enumerate(xs) if srs_fixture.is_square(name, x))


@pytest.mark.parametrize("name", ["pallas_srs", "vesta_srs"])
def test_test_srs_layout_round_trip(request, name, tmp_path):
    """[g, h, {n: [[point]]}] with 65-byte uncompressed points, as srs/test_*.srs"""
    G = request.getfixturevalue(name)
    flag = np.zeros((2048, 1), dtype=np.uint8)
    g65 = np.concatenate([G.g_xy_canon, flag], axis=1)
    h65 = np.concatenate([G.h_xy_canon, [0]]).astype(np.uint8)
    bases = {}
    for k in (10, 0, 3, 1):                      # hash-map order in the reference is arbitrary
        n = 1 << k
        bases[n] = np.concatenate([G.lag_small_canon[n - 1:2 * n - 1], flag[:n]], axis=1).reshape(n, 1, 65)
    path = str(tmp_path / "test.srs")
    srs_file.write_srs(path, srs_file.SrsFile(g=g65, h=h65, lagrange_bases=bases))
    raw = open(path, "rb").read()
    assert raw[:4] == bytes.fromhex("93dc0800") and raw[4:6] == bytes.fromhex("c441")
    back = srs_file.read_srs(path)
    assert not back.compressed and np.array_equal(back.g, g65) and np.array_equal(back.h, h65)
    assert list(back.lagrange_bases) == [1024, 1, 8, 2]
    for n in bases:
        assert np.array_equal(back.lagrange_bases[n], bases[n])
    try:
        import msgpack
    except ImportError:
        return
    obj = msgpack.unpackb(raw, strict_map_key=False)   # an independent decoder reads the same structure
    assert len(obj) == 3 and len(obj[0]) == 2048 and obj[1] == h65.tobytes() and obj[2][8][3][0] == bases[8][3, 0].tobytes()


def test_multi_chunk_bases_and_malformed_input(tmp_path, pallas_srs):
    flag = np.zeros((4, 1), dtype=np.uint8)
    g65 = np.concatenate([pallas_srs.g_xy_canon[:4], flag], axis=1)
    two = np.stack([g65, g65[::-1]], axis=1)        # 4 entries x 2 chunks
    path = str(tmp_path / "chunks.srs")
    srs_file.write_srs(path, srs_file.SrsFile(g=g65, h=g65[0], lagrange_bases={4: two}))
    back = srs_file.read_srs(path)
    assert back.lagrange_bases[4].shape == (4, 2, 65) and np.array_equal(back.lagrange_bases[4], two)
    raw = open(path, "rb").read()
    for bad in (raw[:-1], raw + b"\x00", b"\x94" + raw[1:], raw[:1] + b"\xc0" + raw[2:]):
        p = str(tmp_path / "bad.srs")
        open(p, "wb").write(bad)
        with pytest.raises(ValueError):
            srs_file.read_srs(p)


# poly-commitment/src/precomputed_srs.rs:139-155: rmp-serde of SRS::new(vec![G::generator()], G::generator()), both curves
SRS_ONE_GENERATOR_HEX = ("9291c421010000000000000000000000000000000000000000000000000000000000000000"
                         "c421010000000000000000000000000000000000000000000000000000000000000000")
# curves/src/pasta/curves/pallas.rs:10-15, vesta.rs:10-15
GENERATOR_Y = {"pallas": 12418654782883325593414442427049395787963493412651469444558597405572177144507,
               "vesta": 11426906929455361843568202299992114520848200991084027513389447476559454104162}


def test_one_generator_srs_regression_bytes(orc, tmp_path):
    raw = bytes.fromhex(SRS_ONE_GENERATOR_HEX)
    p = str(tmp_path / "one.srs")
    open(p, "wb").write(raw)
    f = srs_file.read_srs(p)
    assert f.compressed and f.g.shape == (1, 33) and np.array_equal(f.g[0], f.h) and not f.lagrange_bases
    srs_file.write_srs(p, f)
    assert open(p, "rb").read() == raw
    # the oracle's decompression of those 33 bytes is the curve generator of the reference (y = the smaller root: flag 0)
    for name, cid, fid in (("pallas", orc.PALLAS, orc.FP), ("vesta", orc.VESTA, orc.FQ)):
        pt = orc.decompress(cid, f.g.tobytes())[0]
        xy = orc.from_mont(fid, pt.reshape(2, 4))
        assert orc.limbs_to_ints(xy) == [1, GENERATOR_Y[name]]


def test_reader_rejects_corrupted_files_cleanly(tmp_path, vesta_srs):
    """Any truncation or byte flip of a valid file either still parses or raises ValueError — never another exception."""
    import random
    flag = np.zeros((8, 1), dtype=np.uint8)
    g65 = np.concatenate([vesta_srs.g_xy_canon[:8], flag], axis=1)
    bases = {4: np.concatenate([vesta_srs.lag_small_canon[3:7], flag[:4]], axis=1).reshape(4, 1, 65)}
    good = str(tmp_path / "good.srs")
    srs_file.write_srs(good, srs_file.SrsFile(g=g65, h=g65[0], lagrange_bases=bases))
    raw = open(good, "rb").read()
    rng = random.Random(9)
    bad = str(tmp_path / "bad.srs")
    for trial in range(300):
        b = bytearray(raw)
        if trial % 3 == 0:
            b = b[: rng.randrange(len(b))]
        else:
            for _ in range(rng.randrange(1, 4)):
                b[rng.randrange(len(b))] = rng.randrange(256)
        open(bad, "wb").write(bytes(b))
        try:
            srs_file.read_srs(bad)
        except ValueError:
            pass
