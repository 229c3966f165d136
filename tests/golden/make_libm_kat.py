#!/usr/bin/env python3
"""Generate tests/golden/libm_kat.npz: known answers of acosf, sinf, cosf and atan2f from the host's glibc.

Run on a glibc 2.39 x86-64 host whose CPU has FMA - the libm behind the CPU oracle and the golden fixtures, whose bits
csrc/ore_libm.cuh reproduces:
    python tests/golden/make_libm_kat.py
Inputs: every branch threshold of ore_libm.cuh with its +-4-ulp neighbours, signed zeros, denormals, +-1, +-0.5, NaN,
+-inf, the floats nearest k*pi/2 below 120, the floats just below 120, atan2f's special cases in all four quadrants and
50 000 random inputs per function over the arguments the shading code produces (tests/libmkat.py generates them;
the answers to the first 2 000 are stored, all 50 000 as one digest, which keeps the file small).  The table records
the generating host; tests/test_parity_gpu.py holds the device to it and tests/test_lights_textures_cpu.py re-checks it
against the host it runs on.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import libmkat  # noqa: E402

F32, U32 = np.float32, np.uint32


def bits(u):
    return np.array(u, dtype=U32).view(F32)


def around(x, n=4):
    """x (float32) and its n neighbours on either side, both signs"""
    u = np.array([x], F32).view(U32)[0] & U32(0x7FFFFFFF)
    lo = max(0, int(u) - n)
    mags = np.arange(lo, int(u) + n + 1, dtype=np.int64).astype(U32)
    mags = mags[mags <= U32(0x7F800000)]
    return np.concatenate([mags.view(F32), (mags | U32(0x80000000)).view(F32)])


SPECIAL = np.concatenate([
    bits([0x00000000, 0x80000000, 0x00000001, 0x80000001, 0x00400000, 0x807FFFFF, 0x00800000, 0x80800000,
          0x32800000, 0xB2800000, 0x7F7FFFFF, 0xFF7FFFFF, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000, 0x7F800001]),
    np.array([1, -1, 0.5, -0.5, 2, -2, 1e-30, -1e-30, 1e30, -1e30], F32)])


def acos_inputs(rng):
    parts = [SPECIAL]
    for t in (1.0, 0.5, bits([0x32800000])[0]):   # |x| == 1, the |x| < 0.5 split, the tiny-argument return
        parts.append(around(F32(t)))
    parts.append(np.array([1.0000001, -1.0000001, 1.5, -3.0, 1e10], F32))
    return np.concatenate(parts).astype(F32)


def sincos_inputs(rng):
    parts = [SPECIAL]
    # the nominal thresholds and the ones abstop12 (sign, exponent and 3 mantissa bits) actually compares against
    for t in (2.0 ** -12, float.fromhex("0x1.921FB6p-1"), float.fromhex("0x1.9p-1"), 120.0):
        parts.append(around(F32(t)))
    k = np.arange(1, 77)
    kp = (k * np.pi / 2)
    kp = kp[kp < 120]
    for v in kp.astype(F32):                                       # the floats nearest k*pi/2, quadrants past 4 included
        parts.append(around(v))
    below = np.arange(int(np.array([120.0], F32).view(U32)[0]) - 64, int(np.array([120.0], F32).view(U32)[0]), dtype=np.int64)
    b = below.astype(U32).view(F32)                                # 119.99... up to the float below 120
    parts += [b, -b]
    x = np.concatenate(parts).astype(F32)
    # finite |x| >= 120 is CUDA's sinf / cosf on the device (never produced by the shading code): no glibc bits there
    return x[~(np.isfinite(x) & (np.abs(x) >= 120))]


def atan2_inputs(rng):
    ys, xs = [], []
    sp = np.concatenate([SPECIAL, np.array([3.0, -3.0, 1e-38, -1e-38], F32)])
    yy, xx = np.meshgrid(sp, sp, indexing="ij")                    # every quadrant of every special case
    ys.append(yy.ravel())
    xs.append(xx.ravel())
    # x == 1 goes straight to atanf: its thresholds 2^25, 0.4375, 2^-29, 1.1875, 0.6875, 2.4375
    for t in (2.0 ** 25, 0.4375, 2.0 ** -29, 1.1875, 0.6875, 2.4375):
        v = around(F32(t))
        ys.append(v)
        xs.append(np.ones_like(v))
        ys.append(np.ones_like(v))                                 # ... and the same ratios through y / x
        xs.append((1 / v.astype(np.float64)).astype(F32))
    # exponent differences k = 58..63 either way, all four quadrants (k > 60: pi/2; x < 0 and k < -60: 0)
    for k in range(58, 64):
        for s_y in (1, -1):
            for s_x in (1, -1):
                m = rng.uniform(1, 2, 16).astype(F32)
                big, small = (m * F32(2.0 ** (k - 30))).astype(F32), (m[::-1] * F32(2.0 ** -30)).astype(F32)
                ys += [s_y * big, s_y * small]
                xs += [s_x * small, s_x * big]
    return np.concatenate(ys).astype(F32), np.concatenate(xs).astype(F32)


def main():
    desc = libmkat.host_description()
    if not (desc.startswith("glibc 2.39 ") and desc.endswith("x86_64 with FMA")):
        sys.exit(f"this table is glibc 2.39 / x86-64 / FMA; this host is {desc}")
    rng = np.random.default_rng(20260)
    lm = libmkat.host_libm()
    out = {"host": np.array(desc)}
    a = acos_inputs(rng)
    out["acosf_a"], out["acosf_bits"] = a, libmkat.host_eval(lm, "acosf", a).view(U32)
    x = sincos_inputs(rng)
    for op in ("sinf", "cosf"):
        out[op + "_a"], out[op + "_bits"] = x, libmkat.host_eval(lm, op, x).view(U32)
    y, xx = atan2_inputs(rng)
    out["atan2f_a"], out["atan2f_b"], out["atan2f_bits"] = y, xx, libmkat.host_eval(lm, "atan2f", y, xx).view(U32)
    for op in libmkat.OPS:
        ra, rb = libmkat.random_inputs(op)
        r = libmkat.host_eval(lm, op, ra, rb)
        out[op + "_random_head_bits"] = r[:libmkat.RANDOM_STORED].view(U32)
        out[op + "_random_sha256"] = np.array(libmkat.digest(r))
    np.savez_compressed(libmkat.KAT_PATH, **out)
    print(desc, {op: int(out[op + "_a"].size) for op in libmkat.OPS}, "edge inputs +", libmkat.RANDOM_N, "random each,",
          os.path.getsize(libmkat.KAT_PATH), "bytes")


if __name__ == "__main__":
    main()
