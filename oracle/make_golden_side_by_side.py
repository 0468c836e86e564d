"""TEST INFRASTRUCTURE ONLY: writes tests/golden/neo_ref_side_by_side.npz, the inputs and the compiled reference's outputs
(oracle/_ref/libneo_ref.so, the unmodified reference headers compiled in place) of tests/test_oracle.py::test_oracle_vs_compiled_reference,
so that the side-by-side comparison also runs where the reference library is absent.

    python oracle/make_golden_side_by_side.py [OUT]              needs oracle/_ref/libneo_ref.so (`make -C oracle ref`, see oracle/Makefile)
    python oracle/make_golden_side_by_side.py --oracle [OUT]     the oracle's outputs instead: the same arrays only at a commit whose
                                                                 side-by-side test passed against the library, which asserts them bit-identical
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def side_by_side(chk, noise) -> dict:
    """The cases the oracle and the reference are compared on, computed by `chk` (either checker) on inputs drawn by `noise`
    (the oracle's generator, as the comparison has always used), inputs included."""
    g = {}
    for order in range(0, 13):
        g[f"bitrev/{order}"] = chk.bitrev_table(order)
    for order in (1, 4, 9, 13):
        x = noise(1 << order, 21, np.complex64)
        g[f"fft/{order}/x"], g[f"fft/{order}/fwd"] = x, chk.fft(x, -1)
        xr = noise(1 << order, 22, np.float32)
        g[f"rfft/{order}/x"], g[f"rfft/{order}/out"] = xr, chk.rfft(xr)
    g["ir/raw"] = np.stack([noise(700, 31 + c, np.float32) for c in range(2)])
    g["ir/normalized"] = chk.normalize_impulse(g["ir/raw"])
    g["H"] = chk.uniform_partition(g["ir/normalized"], 64)
    g["signal"] = np.stack([noise(64 * 16, 41 + c, np.float32) for c in range(2)])
    for kind in (0, 1, 4):
        g[f"conv/{kind}"] = chk.convolve_blocks(kind, g["H"], g["signal"])
    return g


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    from oracle import pyoracle as po

    args = sys.argv[1:]
    use_oracle = "--oracle" in args
    args = [a for a in args if a != "--oracle"]
    po.build()
    orc = po.oracle()
    chk = orc if use_oracle else po.ref()
    assert chk is not None, "oracle/_ref/libneo_ref.so missing: run `make -C oracle ref` where the reference sources are"
    out = args[0] if args else os.path.join(ROOT, "tests", "golden", "neo_ref_side_by_side.npz")
    g = side_by_side(chk, orc.noise)
    np.savez_compressed(out, **g)
    print(f"wrote {out} from {'the oracle' if use_oracle else chk.path}: {len(g)} arrays, {os.path.getsize(out) / 1024:.1f} KiB")
