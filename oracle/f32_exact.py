"""Exact reference for the text of an f32 as Rust's `f32` Display prints it -- TEST INFRASTRUCTURE ONLY.

Rust (core::fmt -> flt2dec::to_shortest_str, Grisu with the Dragon fallback) prints the fewest significant digits of any
decimal that lies inside the float's rounding interval, and of two such decimals the closer one (the even last digit on a
tie), in positional notation.  The interval is flt2dec::decoder::decode's: half an ulp on either side, except below a
power of two (mantissa field 0, exponent field > 1), where the float below is half as far away; both ends belong to the
interval when the mantissa is even (they read back to this float under round-half-even).

This is a definition, not an algorithm: `display` computes it with fractions.Fraction and shares no code with
csrc/f32_text.h or the oracles.  The matching parse reference is oracle/sam_oracle.py::f32_from_text.
"""
import math
from fractions import Fraction


def _positional(q: int, t: int) -> str:
    """q * 10**t (q > 0) without an exponent, trailing zeros after the point removed."""
    if t >= 0:
        return str(q) + "0" * t
    s = str(q).rjust(1 - t, "0")
    whole, frac = s[:t], s[t:].rstrip("0")
    return whole + "." + frac if frac else whole


def display(bits: int) -> str:
    """Rust's `f32::to_string()` of the f32 with bit pattern `bits`."""
    bits &= 0xFFFFFFFF
    sign, mag = ("-" if bits >> 31 else ""), bits & 0x7FFFFFFF
    if mag > 0x7F800000:
        return "NaN"
    if mag == 0x7F800000:
        return sign + "inf"
    if mag == 0:
        return sign + "0"
    ex, mant = mag >> 23, mag & 0x7FFFFF
    m = mant | 0x800000 if ex else mant
    ulp = Fraction(2) ** ((ex if ex else 1) - 150)
    v = m * ulp
    hi = v + ulp / 2
    lo = v - (ulp / 4 if mant == 0 and ex > 1 else ulp / 2)
    inclusive = m % 2 == 0

    def inside(c):
        return lo < c < hi or (inclusive and (c == lo or c == hi))

    k = math.floor(math.log10(float(v)))              # 10**k <= v < 10**(k + 1), fixed up exactly below
    while Fraction(10) ** k > v:
        k -= 1
    while Fraction(10) ** (k + 1) <= v:
        k += 1
    for n in range(1, 10):                            # 9 significant digits always read back
        t = k - n + 1
        u = Fraction(10) ** t
        q = math.floor(v / u)
        cands = [c for c in (q, q + 1) if inside(c * u)]
        if cands:
            best = min(cands, key=lambda c: (abs(c * u - v), c % 2))
            return sign + _positional(best, t)
    raise AssertionError(f"no decimal of <= 9 digits inside the interval of {bits:#010x}")
