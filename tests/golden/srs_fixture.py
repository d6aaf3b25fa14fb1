"""The golden SRS vectors of one curve (tests/golden/{pallas,vesta}_srs.npz) with the 2^16 compressed generators rebuilt.

The reference's 2^16 generators g[i] (srs/{pallas,vesta}.srs) are not stored: 33 random-looking bytes each would make the
fixtures megabytes.  They are rebuilt from their definition, SRS::create (poly-commitment/src/ipa.rs:751-760): t_i is the
first 248 bits of blake2b-512(u32 big-endian i), read as the reference packs them, and g[i] is the point the Shallue-van de
Woestijne map (groupmap/src/lib.rs, BWParameters with u = 1) sends t_i to.  Two choices the map makes cost a field square
root each, so they are stored instead as one byte per point, `g_sel`: bits 0-1 name the first of the map's three candidate
x-coordinates whose x^3 + 5 is a square, bit 7 is the compressed form's y flag (set: y is the larger of the two roots).
`g_cmp_sha256` is the sha256 of the reference's 2^16 x 33 bytes, so the rebuild is checked against the reference file."""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N_GENERATORS = 1 << 16
MODULUS = {"pallas": 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001,   # base field of each curve
           "vesta": 0x40000000000000000000000000000000224698fc0994a8dd8c46eb2100000001}
# the square root of -3 = -3u^2 that the map's setup takes: the odd one of the two
SQRT_NEG3 = {"pallas": 0x25999506959b74e25955abb8af5563603a3f17a46f5a62923b5abd7bfbfc9573,
             "vesta": 0x0d0334b0507ca51ca23b69b039ee1eb41fda8cfa8f80675e5553a5c0a1541c9f}
COEFF_B = 5


def map_input(i: int) -> int:
    """t_i: bit j of byte k of blake2b-512(i as u32 BE) is bit 8k + j of a 248-bit big-endian bit string"""
    d = hashlib.blake2b(i.to_bytes(4, "big"), digest_size=64).digest()
    return int(format(int.from_bytes(d[:31], "little"), "0248b")[::-1], 2)


def candidate_xs(curve: str, t: int):
    """the map's three candidate x-coordinates for t (u = 1, f(u) = 6)"""
    p, s = MODULUS[curve], SQRT_NEG3[curve]
    u, fu = 1, 1 + COEFF_B
    t2 = t * t % p
    alpha_inv = (t2 + fu) * t2 % p
    alpha = pow(alpha_inv, -1, p) if alpha_inv else 0
    x1 = ((s - u) * pow(2, -1, p) - t2 * t2 % p * alpha % p * s) % p
    x2 = (-u - x1) % p
    tf = (t2 + fu) % p
    x3 = (u - tf * tf % p * (alpha * tf % p) % p * pow(3 * u * u, -1, p)) % p
    return x1, x2, x3


def is_square(curve: str, x: int) -> bool:
    p = MODULUS[curve]
    return pow((x * x * x + COEFF_B) % p, (p - 1) // 2, p) in (0, 1)


def generators(curve: str, sel: np.ndarray) -> np.ndarray:
    """uint8 [len(sel), 33]: g[0..len(sel)) in the compressed form of srs/<curve>.srs (x little-endian, then the y flag byte)"""
    out = np.empty((len(sel), 33), dtype=np.uint8)
    for i, b in enumerate(sel.tolist()):
        x = candidate_xs(curve, map_input(i))[b & 3]
        out[i, :32] = np.frombuffer(x.to_bytes(32, "little"), dtype=np.uint8)
        out[i, 32] = b & 0x80
    return out


def load(curve: str, n: int = N_GENERATORS) -> dict:
    """every array of <curve>_srs.npz, plus g_cmp: uint8 [n, 33], the reference's first n compressed generators"""
    z = dict(np.load(os.path.join(HERE, f"{curve}_srs.npz")))
    z["g_cmp"] = generators(curve, z["g_sel"][:n])
    return z
