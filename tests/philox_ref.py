"""Host reference of the step's own noise (philox_normal4, drvae_b200/csrc/common.cuh).

The integers are recomputed exactly: Philox4x32-10 in uint64 numpy arithmetic on the counter the kernels pack from
(quad q, global row, step, model, draw kind, MC sample l) and the key (the two 32-bit halves of the seed).  The float
steps up to the arguments of the approximate functions are reproduced bit for bit in float32; log, sqrt, sin and cos
are then evaluated in float64, and `allowance` bounds how far the hardware approximations may take each normal from
that value, from the error bounds the PTX ISA documents for them and the fp32 argument reduction of sin / cos.

Test code only: the package never imports this module.
"""
import numpy as np

MASK32 = 0xFFFFFFFF
PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85

# Documented bounds of the approximations philox_normal4 uses (PTX ISA, "Floating Point Instructions"):
E_LG2 = 2.0 ** -22     # lg2.approx.f32: maximum absolute error 2^-22 over the full range (under __logf)
E_SQRT = 2.0 ** -23    # sqrt.approx.f32: maximum relative error 2^-23 over the positive finite range
E_SINCOS = 2.0 ** -20.9  # sin.approx.f32 / cos.approx.f32: maximum absolute error 2^-20.9 over [-pi, pi]
U32 = 2.0 ** -24       # one round-to-nearest fp32 operation: relative error <= 2^-24
LN2_F32 = float(np.float32(np.log(2.0)))  # the constant __logf scales lg2.approx by
TWO_PI_F32 = np.float32(6.283185307179586)
# The angles drawn here lie in [0, 2 pi), beyond the interval of E_SINCOS.  sm_100a evaluates sin.approx / cos.approx as
# one fp32 multiply of the angle by fl32(1 / (2 pi)), rounded toward zero, and a hardware unit periodic in the product
# (in turns).  The product's error, at most 2^-23 relative for the directed rounding plus the constant's relative error,
# moves the result by up to |a| E_REDUCE; so the unit's own error is at most E_SINCOS + pi E_REDUCE (from the bound on
# [-pi, pi]) and the error at angle a at most E_SINCOS + (pi + |a|) E_REDUCE.  Near 2 pi the reduction term is about as
# large as E_SINCOS itself.
E_REDUCE = 2.0 ** -23 + abs(float(np.float32(1 / (2 * np.pi))) * 2 * np.pi - 1)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on arrays of 32-bit counters (any integer dtype) -> four uint64 arrays of 32-bit words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & np.uint64(MASK32) for c in (c0, c1, c2, c3))
    k0 = np.asarray(k0, dtype=np.uint64) & np.uint64(MASK32)
    k1 = np.asarray(k1, dtype=np.uint64) & np.uint64(MASK32)
    m0, m1, sh, mask = np.uint64(PHILOX_M0), np.uint64(PHILOX_M1), np.uint64(32), np.uint64(MASK32)
    for _ in range(10):
        p0 = m0 * c0  # < 2^64: exact
        p1 = m1 * c2
        c0, c1, c2, c3 = (p1 >> sh) ^ c1 ^ k0, p1 & mask, (p0 >> sh) ^ c3 ^ k1, p0 & mask
        k0 = (k0 + np.uint64(PHILOX_W0)) & mask
        k1 = (k1 + np.uint64(PHILOX_W1)) & mask
    return c0, c1, c2, c3


def counter(q, grow, step, model, seg, l):
    """The counter philox_normal4 packs: {q | (grow >> 32) << 24, (uint32) grow, step, model | seg << 20 | l << 24}."""
    q, grow, step, model, seg, l = (np.asarray(a, dtype=np.uint64) for a in (q, grow, step, model, seg, l))
    mask = np.uint64(MASK32)
    c0 = (q | ((grow >> np.uint64(32)) << np.uint64(24))) & mask
    c1 = grow & mask
    c2 = step & mask
    c3 = (model | (seg << np.uint64(20)) | (l << np.uint64(24))) & mask
    return c0, c1, c2, c3


def _u_open(c):
    """(c + 1.0f) * 2^-32 in float32: uint32 -> float (one rounding), + 1 (one rounding), exact power-of-two scaling."""
    f = c.astype(np.float64).astype(np.float32)
    return ((f + np.float32(1.0)) * np.float32(2.0 ** -32)).astype(np.float32)


def _u_closed(c):
    return (c.astype(np.float64).astype(np.float32) * np.float32(2.0 ** -32)).astype(np.float32)


def normals(seed, step, model, seg, l, grow, q):
    """The four normals of each quad -> (z [..., 4] float64 reference, allowance [..., 4]).

    Arguments broadcast against each other.  Up to log / sqrt / sin / cos the float32 steps of the kernel are exact
    here; those four are float64, and `allowance` is the documented worst case of the kernel's approximations."""
    seed = int(seed)
    c = philox4x32_10(*counter(q, grow, step, model, seg, l), seed & MASK32, seed >> 32)
    u0 = np.minimum(_u_open(c[0]), np.float32(1.0))
    u2 = np.minimum(_u_open(c[2]), np.float32(1.0))
    a1 = (TWO_PI_F32 * _u_closed(c[1])).astype(np.float32)
    a3 = (TWO_PI_F32 * _u_closed(c[3])).astype(np.float32)
    z, allow = [], []
    for u, a in ((u0, a1), (u2, a3)):
        r_lo, r, r_hi = _radius(u)
        a = a.astype(np.float64)
        e_trig = E_SINCOS + (np.pi + a) * E_REDUCE
        for f in (np.cos, np.sin):
            zz, aa = _product(r_lo, r, r_hi, f(a), e_trig)
            z.append(zz)
            allow.append(aa)
    return np.stack(z, axis=-1), np.stack(allow, axis=-1)


def _radius(u):
    """sqrt(-2 ln u) and the interval the kernel's radius lies in.

    t = -2 * (lg2.approx(u) * ln2_f32): the log error E_LG2 scaled by ln 2, the difference of the fp32 constant from
    ln 2, and one rounding each for the two multiplies.  Propagated through sqrt as the interval
    [sqrt(max(t - d, 0)), sqrt(t + d)] (a first-order bound fails where t is near 0, u near 1), then the relative
    error of sqrt.approx."""
    lg = np.log2(u.astype(np.float64))
    t = -2.0 * np.log(2.0) * lg
    d = 2.0 * (E_LG2 * LN2_F32 + np.abs(lg) * abs(LN2_F32 - np.log(2.0))) + 2.0 * U32 * (t + 2.0 * E_LG2)
    lo = np.sqrt(np.maximum(t - d, 0.0)) * (1.0 - E_SQRT)
    hi = np.sqrt(t + d) * (1.0 + E_SQRT)
    return lo, np.sqrt(t), hi


def _product(r_lo, r, r_hi, cs, e_trig):
    """z = fl32(r * cos) with r in [r_lo, r_hi] and the approximate cos within e_trig: the bilinear product takes its
    extremes at the corners; plus one rounding of the product."""
    ref = r * cs
    worst = np.zeros_like(ref)
    big = np.zeros_like(ref)
    for rr in (r_lo, r_hi):
        for cc in (cs - e_trig, cs + e_trig):
            p = rr * cc
            worst = np.maximum(worst, np.abs(p - ref))
            big = np.maximum(big, np.abs(p))
    return ref, worst + U32 * big
