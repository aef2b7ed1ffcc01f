"""Accuracy of angle_from_cos_sin2 (csrc/hmp_kernels.cu), the FP32 angle of the sweep's static-object and people loops, checked
on the CPU against math.asin / math.acos on >= 10^6 (cosine, sine) pairs: a uniform sweep of the angle over [0, pi], dense runs
around the octant boundaries pi/4 and 3 pi/4, and the exact edge cases c = +-1, s = 0, c = +-0, s = |c|.

The routine is emulated operation by operation in FP32: every fused multiply-add as the exact FP64 product plus the addend,
rounded to FP64 and then to FP32 (the double rounding can differ from the device's single rounding by one FP32 ulp in rare
ties, far below the bar). The reference is the angle the routine defines for its inputs, in FP64: asin(s) in front
(s <= |c|, c >= 0), pi - asin(s) behind (s <= |c|, c < 0), acos(c) otherwise. The routine returns the angle up to its sign (its
callers square it), so |result| is compared.

Bar: 1e-7 absolute plus one FP32 ulp of the result (a result near pi cannot be closer than half an ulp, 1.2e-7, and the FP32
constants pi and pi/2 are themselves 8.7e-8 and 4.4e-8 off), and no larger maximum error than the routine it replaced (select-
based octant, degree-8 polynomial, also measured here) on either half of [0, pi].
usage: python tools/check_angle_fp32.py"""
import math
import sys

import numpy as np

f32 = np.float32
PI_F = f32(math.pi)


def fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + np.asarray(c, dtype=np.float64)).astype(f32)


# coefficients of asin(z) / z in z^2, highest degree first, as in the kernel
NEW = [1.305062175e-01, -1.288138181e-01, 1.043007821e-01, 5.871396512e-03, 4.867245629e-02, 7.465469837e-02, 1.666798294e-01,
       9.999998808e-01]
OLD = [1.448995462e-01, -1.801251085e-01, 1.457034517e-01, -2.460549290e-02, 4.040429929e-02, 4.341339492e-02, 7.508057529e-02,
       1.666642890e-01, 1.000000020e+00]


def horner(coef, q):
    p = np.full_like(q, f32(coef[0]))
    for k in coef[1:]:
        p = fma(p, q, f32(k))
    return p


def angle_new(c, s):
    d = (np.abs(c) - s).astype(f32)
    hi = np.signbit(d)
    z = np.where(hi, c, s)
    base = np.where(hi, f32(-0.5) * PI_F, np.where(np.signbit(c), -PI_F, f32(0.0))).astype(f32)
    q = (z * z).astype(f32)
    return fma(z, horner(NEW, q), base)


def angle_old(c, s):
    lo = s <= np.abs(c)
    z = np.where(lo, s, c)
    r = (z * horner(OLD, (z * z).astype(f32))).astype(f32)
    return np.where(lo, np.where(c < 0, (PI_F - r).astype(f32), r), (f32(0.5 * math.pi) - r).astype(f32))


def reference(c, s):
    c64, s64 = c.astype(np.float64), s.astype(np.float64)
    lo = s64 <= np.abs(c64)
    a_front = np.arcsin(np.minimum(s64, 1.0))
    return np.where(lo, np.where(c64 < 0, math.pi - a_front, a_front), np.arccos(np.clip(c64, -1.0, 1.0)))


def inputs():
    rng = np.random.default_rng(0)
    th = [np.linspace(0.0, math.pi, 1_000_001), rng.uniform(0.0, math.pi, 500_000)]
    for b in (math.pi / 4, 3 * math.pi / 4, math.pi / 2):   # octant boundaries and the right angle, dense
        th.append(b + np.linspace(-1e-3, 1e-3, 100_001))
    th = np.concatenate(th)
    c, s = np.cos(th).astype(f32), np.abs(np.sin(th)).astype(f32)
    # the same angles from a cosine with the sine derived in FP32 (inputs that are not exactly on the unit circle)
    c2 = rng.uniform(-1.0, 1.0, 500_000).astype(f32)
    s2 = np.sqrt(np.maximum(f32(1) - c2 * c2, f32(0))).astype(f32)
    h = f32(math.sqrt(0.5))
    edge_c = np.array([1, -1, 0, -0.0, h, -h, h, -h, np.nextafter(h, f32(1)), np.nextafter(h, f32(0))], dtype=f32)
    edge_s = np.array([0, 0, 1, 1, h, h, np.nextafter(h, f32(1)), np.nextafter(h, f32(1)), h, h], dtype=f32)
    return np.concatenate([c, c2, edge_c]), np.concatenate([s, s2, edge_s])


def main():
    c, s = inputs()
    ref = reference(c, s)
    bar = 1e-7 + np.spacing(ref.astype(f32)).astype(np.float64)
    front, back = ref <= math.pi / 2, ref > math.pi / 2
    worst_half = {}
    for name, fn in (("new", angle_new), ("previous", angle_old)):
        a = np.abs(fn(c, s).astype(np.float64))
        err = np.abs(a - ref)
        worst_half[name] = (err[front].max(), err[back].max())
        worst = int(np.argmax(err - bar))
        print(f"{name:7s} {len(c)} points: max |error| {err[front].max():.3e} on [0, pi/2], {err[back].max():.3e} on (pi/2, pi]; "
              f"worst against the bar at c = {c[worst]!r}, s = {s[worst]!r}: {err[worst]:.3e} (bar {bar[worst]:.3e})")
        if name == "new":
            ok = bool(np.all(err <= bar))
    ok = ok and all(n <= o for n, o in zip(worst_half["new"], worst_half["previous"]))
    print("PASS" if ok else "FAIL")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
