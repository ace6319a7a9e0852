#!/usr/bin/env python3
"""Record what the reference's own halfutils.c / bitutils.c (oracle/_ref/libpgvref.so, built by oracle.build() when
the pgvector source tree is present) return on fixed inputs, into tests/golden/ref_kernels.npz.

    python tests/golden/make_ref_kernels.py

tests/test_oracle_golden.py compares the oracle's restatement against these stored outputs, so the comparison runs
wherever the tests run, with or without the pgvector sources.  Inputs are stored beside the outputs.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle as O  # noqa: E402
from tests.util import f32_to_half_bits  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_kernels.npz")
HALF_DIMS = (1, 3, 8, 9, 64, 100, 768, 1537)
BIT_LENGTHS = (0, 1, 7, 8, 52, 63, 64, 65, 513, 1024, 4099)


def main():
    O.build()
    R = O.ref()
    if R is None:
        sys.exit("oracle/_ref/libpgvref.so was not built: the pgvector source tree is needed")
    out = {}
    # float -> half (RNE) on random values and the edge cases around the half range; half -> float on every 7th pattern
    rng = np.random.default_rng(0)
    xs = np.concatenate([
        rng.standard_normal(2000).astype(np.float32) * 10,
        np.float32([0, -0.0, 1, -1, 65504, 65520, 65519.99, 1e-8, 5.96e-8, 2.98e-8, 2.9802322e-8, 6.1e-5, 6.0975552e-5,
                    1e5, -1e5, np.inf, -np.inf, 0.1, 0.33325195, 1.0009766, 1.00048828125, 1.0014648]),
        (rng.standard_normal(500) * 1e-6).astype(np.float32),
    ])
    out["f2h_in"] = xs
    out["f2h_out"] = np.array([R.ref_float_to_half(float(x)) for x in xs], dtype=np.uint16)
    out["h2f_in"] = np.arange(0, 65536, 7, dtype=np.uint16)
    out["h2f_out"] = np.array([R.ref_half_to_float(int(h)) for h in out["h2f_in"]], dtype=np.float32)
    # half distance kernels
    rng = np.random.default_rng(1)
    for dim in HALF_DIMS:
        a = f32_to_half_bits(rng.standard_normal(dim))
        b = f32_to_half_bits(rng.standard_normal(dim))
        pa, pb = a.ctypes.data, b.ctypes.data
        out[f"half_a_{dim}"], out[f"half_b_{dim}"] = a, b
        out[f"half_out_{dim}"] = np.array([R.ref_half_l2sq(dim, pa, pb), R.ref_half_ip(dim, pa, pb),
                                           R.ref_half_l1(dim, pa, pb), R.ref_half_cos(dim, pa, pb)], dtype=np.float64)
    # bit distance kernels (padding bits of the last byte cleared, as varbit stores them)
    for nbits in BIT_LENGTHS:
        nbytes = (nbits + 7) // 8
        a = rng.integers(0, 256, size=max(nbytes, 1), dtype=np.uint8)[:nbytes].copy()
        b = rng.integers(0, 256, size=max(nbytes, 1), dtype=np.uint8)[:nbytes].copy()
        if nbits % 8 and nbytes:
            mask = (0xFF << (8 - nbits % 8)) & 0xFF
            a[-1] &= mask
            b[-1] &= mask
        pa = a.ctypes.data if nbytes else None
        pb = b.ctypes.data if nbytes else None
        out[f"bit_a_{nbits}"], out[f"bit_b_{nbits}"] = a, b
        out[f"bit_hamming_{nbits}"] = np.uint64(R.ref_bit_hamming(nbytes, pa, pb))
        out[f"bit_jaccard_{nbits}"] = np.float64(R.ref_bit_jaccard(nbytes, pa, pb))
    np.savez_compressed(OUT, **out)
    print(f"{OUT}: {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
