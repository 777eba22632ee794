"""CPU emulation of the 3-pass split-tf32 dot products of the DCN (forward and backward GEMMs): how the error floor of
the MREFSR_DCN_TF32X3 mode depends on how the tensor core rounds its fp32 accumulator.

    python tools/dcn_x3_accum_sim.py [--outputs N]

Each output is a dot product of length K (K = 9 * C in the forward).  The operands are split as the kernels split
them (hi = v rounded to tf32 with the low bits cleared, lo = tf32(v - hi)); one MMA adds the exact sum of 8 products
of one pass (lo.hi, hi.lo, hi.hi, in that order) to the fp32 accumulator, which is rounded either to nearest (RN) or
toward zero (RZ) after each add.  The error is reported as the tests measure it: max |out - exact| / max |exact| over
all outputs.  With RN it grows like sqrt(K); with RZ the roundings all point the same way and it grows like K.
The tf32 (one-pass) mode's error is shown for scale."""
import argparse

import numpy as np


def tf32_hi(v):
    b = v.astype(np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def to_fp32(v, mode):
    f = v.astype(np.float32)
    if mode == 'rz':                   # step back toward zero where round-to-nearest went past v
        over = np.abs(f.astype(np.float64)) > np.abs(v)
        f[over] = np.nextafter(f[over], np.float32(0))
    return f


def dot_emulated(a, b, mode, passes):
    """a [N, K], b [K] fp32 -> fp32 [N] as the MMA sequence would accumulate it."""
    ah, bh = tf32_hi(a), tf32_hi(b)
    al, bl = tf32_hi(a - ah), tf32_hi(b - bh)
    terms = {'lo.hi': (al, bh), 'hi.lo': (ah, bl), 'hi.hi': (ah, bh)}
    acc = np.zeros(a.shape[0], np.float32)
    for k0 in range(0, a.shape[1], 8):
        for p in passes:
            x, y = terms[p]
            s = (x[:, k0:k0 + 8].astype(np.float64) * y[k0:k0 + 8].astype(np.float64)).sum(1)   # exact for 8 products
            acc = to_fp32(acc.astype(np.float64) + s, mode)
    return acc


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--outputs', type=int, default=4096)
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    print('%6s %6s  %-22s %-22s %s' % ('C', 'K', 'x3, RN accumulator', 'x3, RZ accumulator', 'tf32 (one pass), RZ'))
    for c in (64, 128, 256):
        k = 9 * c
        # bilinear samples of unit-variance features times a mask in (0, 1), and weights of scale (9 C)^-1/2, as the tests
        a = (rng.standard_normal((args.outputs, k)) * rng.random((args.outputs, k))).astype(np.float32)
        b = (rng.standard_normal(k) * k ** -0.5).astype(np.float32)
        exact = a.astype(np.float64) @ b.astype(np.float64)

        def err(out):
            return float(np.abs(out - exact).max() / np.abs(exact).max())
        e_rn = err(dot_emulated(a, b, 'rn', ('lo.hi', 'hi.lo', 'hi.hi')))
        e_rz = err(dot_emulated(a, b, 'rz', ('lo.hi', 'hi.lo', 'hi.hi')))
        e_1 = err(dot_emulated(a, b, 'rz', ('hi.hi',)))
        print('%6d %6d  %-22.3g %-22.3g %.3g' % (c, k, e_rn, e_rz, e_1))


if __name__ == '__main__':
    main()
