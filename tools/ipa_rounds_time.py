"""Wall time of the 16 folding rounds of a 2^16 IPA opening (SRS::open, ipa.rs:929-1007) through the C ABI: per round one lr()
(two table MSMs + two inner products) and one fold(); challenges are arbitrary field elements (the sponge is the caller's)."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import proof_systems_b200 as zk  # noqa: E402
from bench import splitmix64_limbs  # noqa: E402

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden"))
import srs_fixture  # noqa: E402


def main():
    z = srs_fixture.load("pallas")
    ctx = zk.Context(0)
    g = ctx.decompress_points(zk.PALLAS, z["g_cmp"])
    n = g.shape[0]
    k = n.bit_length() - 1
    bases = ctx.upload_bases(zk.PALLAS, g)
    a = splitmix64_limbs(1, n)   # used as Montgomery representations: any residues do
    b = splitmix64_limbs(2, n)
    us = splitmix64_limbs(3, 2 * k)
    for rep in range(3):
        t0 = time.perf_counter()
        r = zk.IpaRounds(ctx, bases, a, b)
        t1 = time.perf_counter()
        for j in range(k):
            r.lr()
            r.fold(us[2 * j], us[2 * j + 1])
        sg = r.sg()
        a0, b0 = r.state()
        t2 = time.perf_counter()
        r.close()
        print(f"rep {rep}: n = 2^{k}: upload {1e3 * (t1 - t0):.2f} ms, {k} rounds + sg {1e3 * (t2 - t1):.2f} ms")
    ctx.close()


if __name__ == "__main__":
    main()
