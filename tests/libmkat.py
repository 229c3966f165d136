"""The device libm's known answers (tests/golden/libm_kat.npz, written by tests/golden/make_libm_kat.py): the bits glibc
2.39 on an FMA-capable x86-64 host returns for the inputs of acosf, sinf, cosf and atan2f that matter to
csrc/ore_libm.cuh, and this host's libm called on the same inputs.  TEST INFRASTRUCTURE ONLY.

The table holds two parts per function:
  * the edge inputs (branch thresholds and their neighbours, special values; stored with their answers), and
  * RANDOM_N random inputs over the arguments the shading code produces, generated here from a counter-based hash
    (integer arithmetic and IEEE float operations only: the same inputs on every host and numpy version).  The answers
    to the first RANDOM_STORED of them are stored bit for bit, so that a mismatch can be located; all RANDOM_N answers
    are stored as one SHA-256 digest, which keeps the file small."""
import ctypes as C
import ctypes.util
import hashlib
import os
import platform

import numpy as np

KAT_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "libm_kat.npz")
OPS = ("acosf", "sinf", "cosf", "atan2f")
RANDOM_N = 50000
RANDOM_STORED = 2000
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def host_libm():
    lm = C.CDLL(ctypes.util.find_library("m") or "libm.so.6")
    for n in ("cosf", "sinf", "acosf"):
        getattr(lm, n).restype = C.c_float
        getattr(lm, n).argtypes = [C.c_float]
    lm.atan2f.restype = C.c_float
    lm.atan2f.argtypes = [C.c_float, C.c_float]
    return lm


def host_eval(lm, op, a, b=None):
    """this host's libm on float32 inputs (atan2f: a = y, b = x), float32 results"""
    f = getattr(lm, op)
    if op == "atan2f":
        return np.array([f(float(p), float(q)) for p, q in zip(a, b)], dtype=np.float32)
    return np.array([f(float(v)) for v in a], dtype=np.float32)


def glibc_version():
    try:
        fn = C.CDLL(None).gnu_get_libc_version
        fn.restype = C.c_char_p
        return fn().decode()
    except (AttributeError, OSError):
        return ""


def cpu_has_fma():
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags"):
                    return " fma " in line + " "
    except OSError:
        pass
    return False


def host_description():
    return f"glibc {glibc_version() or 'none'} on {platform.machine()}" + (" with FMA" if cpu_has_fma() else " without FMA")


# ---- the random inputs ------------------------------------------------------------------------------------------------

def _uniform(stream, n, lo, hi):
    """n float32 values in [lo, hi): splitmix64 of (stream, index), its top 53 bits as a double in [0, 1), then
    lo + (hi - lo) * u rounded to float32 (exact double operations: no libm involved)"""
    x = np.arange(n, dtype=np.uint64) + np.uint64((stream * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF)
    for sh, mul in ((30, 0xBF58476D1CE4E5B9), (27, 0x94D049BB133111EB)):
        x = ((x ^ (x >> np.uint64(sh))) * np.uint64(mul)) & _M64
    x ^= x >> np.uint64(31)
    u = (x >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    return (lo + (hi - lo) * u).astype(np.float32)


def random_inputs(op):
    """(a, b) of the RANDOM_N random inputs of op (b is None but for atan2f)"""
    if op == "acosf":   # unit-vector components, and both ends of the domain
        a = np.concatenate([_uniform(1, 40000, -1, 1), (1 - _uniform(2, 5000, 0, 1e-3)).astype(np.float32),
                            (_uniform(3, 5000, 0, 1e-3) - 1).astype(np.float32)])
        return a, None
    if op in ("sinf", "cosf"):   # 2*dot(unit, unit), acosf results, camera angles; the whole |x| < 120 range
        x = np.concatenate([_uniform(4, 30000, -4, 4), _uniform(5, 20000, -120, 120)])
        return np.where(np.abs(x) < 120, x, np.float32(0)).astype(np.float32), None
    # atan2f: (z, x) components of unit normals, normalised in float32 (IEEE sqrt and division only)
    v = [_uniform(6 + k, RANDOM_N, -1, 1) for k in range(3)]
    n2 = (v[0] * v[0] + v[1] * v[1]).astype(np.float32) + v[2] * v[2]
    length = np.sqrt(n2.astype(np.float32)).astype(np.float32)
    length = np.where(length > 0, length, np.float32(1))
    return (v[2] / length).astype(np.float32), (v[0] / length).astype(np.float32)


def digest(results):
    """SHA-256 of float32 result bits, every NaN counted as the same NaN (see mismatches)"""
    r = np.ascontiguousarray(results, dtype=np.float32).copy()
    bits = r.view(np.uint32)
    bits[np.isnan(r)] = 0x7FC00000
    return hashlib.sha256(bits.tobytes()).hexdigest()


# ---- the table ----------------------------------------------------------------------------------------------------------

def load():
    """{op: dict(a, b, bits, ra, rb, rbits_head, rdigest)} and the generating host's description; a / b / bits are the
    edge inputs and answers, ra / rb the random inputs, rbits_head the answers to the first RANDOM_STORED of them and
    rdigest the digest of all their answers"""
    d = np.load(KAT_PATH)
    table = {}
    for op in OPS:
        ra, rb = random_inputs(op)
        table[op] = dict(a=d[op + "_a"], b=d[op + "_b"] if op == "atan2f" else None, bits=d[op + "_bits"], ra=ra, rb=rb,
                         rbits_head=d[op + "_random_head_bits"], rdigest=str(d[op + "_random_sha256"]))
    return table, str(d["host"])


def mismatches(got, want_bits):
    """indices where float32 results `got` differ from the stored bits; a stored NaN asks for any NaN (its sign and
    payload are the x87/SSE default, not part of what the shading code reads)"""
    g = np.ascontiguousarray(got, dtype=np.float32).view(np.uint32)
    want = want_bits.view(np.float32)
    ok = (g == want_bits) | (np.isnan(want) & np.isnan(got))
    return np.nonzero(~ok)[0]


def check(op, t, evaluate):
    """problems of `evaluate(a, b) -> float32 results` against the table entry t of op; empty when it reproduces it"""
    problems = []
    got = evaluate(t["a"], t["b"])
    bad = mismatches(got, t["bits"])
    if bad.size:
        problems.append((op, "edge inputs", int(bad.size), [(float(t["a"][i]), None if t["b"] is None else float(t["b"][i]),
                                                            hex(int(got.view(np.uint32)[i])), hex(int(t["bits"][i])))
                                                           for i in bad[:6]]))
    rgot = evaluate(t["ra"], t["rb"])
    bad = mismatches(rgot[:RANDOM_STORED], t["rbits_head"])
    if bad.size:
        problems.append((op, f"first {RANDOM_STORED} random inputs", int(bad.size),
                         [float(t["ra"][i]) for i in bad[:6]]))
    if digest(rgot) != t["rdigest"]:
        problems.append((op, f"digest of all {RANDOM_N} random answers differs"))
    return problems


def host_reproduces(lm=None):
    """True when this host's libm returns the stored answers for every entry (the oracle can then be matched exactly)"""
    lm = lm or host_libm()
    table, _ = load()
    return not any(check(op, t, lambda a, b, op=op: host_eval(lm, op, a, b)) for op, t in table.items())
