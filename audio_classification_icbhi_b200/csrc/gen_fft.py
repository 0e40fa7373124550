#!/usr/bin/env python3
"""Emits straight-line, register-resident radix-2 DIT FFT kernels (fft_gen.cuh).

Every index and twiddle is a compile-time literal, so nvcc keeps whole arrays in registers.
Three flavours of the same forward transform (sign e^{-2 pi i nk/N}), natural order in and out:

  lm_fft{8,16,32}(float xr[N], float xi[N])
      scalar reference flavour (used by the CPU tests and as documentation of the op count).

  lm_fft32_aos(lm_f2 z[32])
      one complex point per 64-bit register (lo = re, hi = im), packed fp32x2 arithmetic:
      every butterfly is 2 FADD2 or 3 FFMA2 -- half the issue slots of the scalar flavour.
      Used for the first (lane-local) FFT, whose input arrives from shared memory as float2.

  lm_fft32_aos_from2(lm_f2 z[32])
      the same network minus its first stage: the kernel computes z[r] +- z[r+16] itself, fused
      with the Hann window (hann[n + n_fft/2] = 1 - hann[n], so one window load serves both inputs).

  lm_fft32_soa(const lm_f2 pr[16], const lm_f2 pi[16], float xr[32], float xi[32])
      input pr[m] = (re x[2m], re x[2m+1]), pi[m] likewise -- what the LDS.128 reads of the
      32x32 transpose deliver.  In DIT order those two points share every twiddle of stages 1-4
      (they are the even- and odd-sample 16-point sub-transforms), so stages 1-4 run packed with
      broadcast constants; stage 5 combines the halves of each register in scalar code.

  lm_fft16x2_soa / lm_fft8x4_soa(const lm_f2 pr[16], const lm_f2 pi[16], float xr[32], float xi[32])
      the same layout cut into 2 independent 16-point or 4 independent 8-point transforms (the
      second stage of the 512- and 256-point FFTs): transform b reads pr/pi[b n/2 ..] and writes
      xr/xi[b n ..]; all stages but the last run packed.

Non-trivial butterflies use the 6-FMA (3 packed) Linzer-Feig form with the tangent
(|c| >= |s|) or cotangent (|c| < |s|) ratio so that |ratio| <= 1:

    w = c - i s,  t = s/c:   b~ = (br + t bi, bi - t br)        a +- c b~
    w = c - i s,  t = c/s:   b^ = (br - t bi, bi + t br)        a +- s (b^i, -b^r)

The text only uses the helpers of lm_f2.cuh, which are PTX f32x2 ops under nvcc and plain C
under gcc: tests/test_fft_codegen.py compiles this very file with gcc and checks it against numpy.

Usage:  python gen_fft.py > fft_gen.cuh
"""
import math


def bitrev(i: int, bits: int) -> int:
    r = 0
    for _ in range(bits):
        r = (r << 1) | (i & 1)
        i >>= 1
    return r


def lit(x: float) -> str:
    return f"{x:.9e}f"


def twiddle_kind(j: int, m: int):
    """('one'|'mi'|'tan'|'cot', c, s, t) for w = exp(-2 pi i j / m)."""
    c = math.cos(2 * math.pi * j / m)
    s = math.sin(2 * math.pi * j / m)
    if j == 0:
        return "one", c, s, 0.0
    if 4 * j == m:
        return "mi", c, s, 0.0
    if abs(c) >= abs(s):
        return "tan", c, s, s / c
    return "cot", c, s, c / s


# --------------------------------------------------------------------------------------
def gen_scalar(n: int) -> str:
    bits = n.bit_length() - 1
    out, ops, tmp = [], 0, 0
    emit = out.append
    emit(f"LM_HD LM_INLINE void lm_fft{n}(float (&xr)[{n}], float (&xi)[{n}]) {{")
    cur = [(f"xr[{bitrev(i, bits)}]", f"xi[{bitrev(i, bits)}]") for i in range(n)]
    for s in range(1, bits + 1):
        m, half = 1 << s, 1 << (s - 1)
        for k in range(0, n, m):
            for j in range(half):
                ia, ib = k + j, k + j + half
                (ar, ai), (br, bi) = cur[ia], cur[ib]
                p = f"t{tmp}"
                tmp += 1
                kind, c, sn, t = twiddle_kind(j, m)
                if kind == "one":
                    emit(f"  const float {p}ar = {ar} + {br}, {p}ai = {ai} + {bi};")
                    emit(f"  const float {p}br = {ar} - {br}, {p}bi = {ai} - {bi};")
                    ops += 4
                elif kind == "mi":
                    emit(f"  const float {p}ar = {ar} + {bi}, {p}ai = {ai} - {br};")
                    emit(f"  const float {p}br = {ar} - {bi}, {p}bi = {ai} + {br};")
                    ops += 4
                elif kind == "tan":
                    emit(f"  const float {p}ur = fmaf({lit(t)}, {bi}, {br}), {p}ui = fmaf({lit(-t)}, {br}, {bi});")
                    emit(f"  const float {p}ar = fmaf({lit(c)}, {p}ur, {ar}), {p}ai = fmaf({lit(c)}, {p}ui, {ai});")
                    emit(f"  const float {p}br = fmaf({lit(-c)}, {p}ur, {ar}), {p}bi = fmaf({lit(-c)}, {p}ui, {ai});")
                    ops += 6
                else:
                    emit(f"  const float {p}ur = fmaf({lit(-t)}, {bi}, {br}), {p}ui = fmaf({lit(t)}, {br}, {bi});")
                    emit(f"  const float {p}ar = fmaf({lit(sn)}, {p}ui, {ar}), {p}ai = fmaf({lit(-sn)}, {p}ur, {ai});")
                    emit(f"  const float {p}br = fmaf({lit(-sn)}, {p}ui, {ar}), {p}bi = fmaf({lit(sn)}, {p}ur, {ai});")
                    ops += 6
                cur[ia] = (f"{p}ar", f"{p}ai")
                cur[ib] = (f"{p}br", f"{p}bi")
    for i in range(n):
        emit(f"  xr[{i}] = {cur[i][0]}; xi[{i}] = {cur[i][1]};")
    emit("}")
    emit(f"// lm_fft{n}: {ops} scalar float ops")
    return "\n".join(out)


# --------------------------------------------------------------------------------------
def gen_aos(n: int, first_stage: int = 1) -> str:
    """Packed complex (re, im) per register.  first_stage = 2: z[] already holds the results of the
    first butterfly stage (z[r] +- z[r + n/2] in place) -- the caller fused it with the window."""
    bits = n.bit_length() - 1
    out, ops, tmp = [], 0, 0
    emit = out.append
    name = f"lm_fft{n}_aos" if first_stage == 1 else f"lm_fft{n}_aos_from{first_stage}"
    emit(f"LM_HD LM_INLINE void {name}(lm_f2 (&z)[{n}]) {{")
    cur = [f"z[{bitrev(i, bits)}]" for i in range(n)]
    for s in range(first_stage, bits + 1):
        m, half = 1 << s, 1 << (s - 1)
        for k in range(0, n, m):
            for j in range(half):
                ia, ib = k + j, k + j + half
                a, b = cur[ia], cur[ib]
                p = f"c{tmp}"
                tmp += 1
                kind, c, sn, t = twiddle_kind(j, m)
                if kind == "one":
                    emit(f"  const lm_f2 {p}a = lm_add2({a}, {b}), {p}b = lm_sub2({a}, {b});")
                    ops += 2
                elif kind == "mi":   # w b = -i b = (bi, -br)
                    emit(f"  const lm_f2 {p}a = lm_add2({a}, lm_mul_mi({b})), {p}b = lm_sub2({a}, lm_mul_mi({b}));")
                    ops += 2
                elif kind == "tan":  # b~ = b + t (bi, -br);  a +- c b~
                    emit(f"  const lm_f2 {p}u = lm_fma2(lm_swap({b}), lm_pack({lit(t)}, {lit(-t)}), {b});")
                    emit(f"  const lm_f2 {p}a = lm_fma2({p}u, lm_bcast({lit(c)}), {a}), "
                         f"{p}b = lm_fma2({p}u, lm_bcast({lit(-c)}), {a});")
                    ops += 3
                else:                # b^ = b + t (-bi, br);  a +- s (b^i, -b^r)
                    emit(f"  const lm_f2 {p}u = lm_fma2(lm_swap({b}), lm_pack({lit(-t)}, {lit(t)}), {b});")
                    emit(f"  const lm_f2 {p}a = lm_fma2(lm_swap({p}u), lm_pack({lit(sn)}, {lit(-sn)}), {a}), "
                         f"{p}b = lm_fma2(lm_swap({p}u), lm_pack({lit(-sn)}, {lit(sn)}), {a});")
                    ops += 3
                cur[ia], cur[ib] = f"{p}a", f"{p}b"
    for i in range(n):
        emit(f"  z[{i}] = {cur[i]};")
    emit("}")
    emit(f"// {name}: {ops} packed f32x2 ops")
    return "\n".join(out)


# --------------------------------------------------------------------------------------
def gen_soa(n: int = 32) -> str:
    """32 // n independent n-point transforms of the 32 points one lane holds after the transpose:
    transform b reads pr/pi[b n/2 .. b n/2 + n/2 - 1] and writes xr/xi[b n .. b n + n - 1].
    Stages 1 .. log2(n)-1 on (even-sample, odd-sample) register pairs, the last stage scalar."""
    count, h = 32 // n, n // 2
    hbits = h.bit_length() - 1
    name = "lm_fft32_soa" if n == 32 else f"lm_fft{n}x{count}_soa"
    out, ops2, ops1, tmp = [], 0, 0, 0
    emit = out.append
    emit(f"LM_HD LM_INLINE void {name}(const lm_f2 (&pr)[16], const lm_f2 (&pi)[16], "
         "float (&xr)[32], float (&xi)[32]) {")
    for b in range(count):
        # DIT-(n/2) array A[i] = P[bitrev(i)], each entry a (re pair, im pair)
        cur = [(f"pr[{b * h + bitrev(i, hbits)}]", f"pi[{b * h + bitrev(i, hbits)}]") for i in range(h)]
        for s in range(1, hbits + 1):
            m, half = 1 << s, 1 << (s - 1)
            for k in range(0, h, m):
                for j in range(half):
                    ia, ib = k + j, k + j + half
                    (ar, ai), (br, bi) = cur[ia], cur[ib]
                    p = f"s{tmp}"
                    tmp += 1
                    kind, c, sn, t = twiddle_kind(j, m)
                    if kind == "one":
                        emit(f"  const lm_f2 {p}ar = lm_add2({ar}, {br}), {p}ai = lm_add2({ai}, {bi});")
                        emit(f"  const lm_f2 {p}br = lm_sub2({ar}, {br}), {p}bi = lm_sub2({ai}, {bi});")
                        ops2 += 4
                    elif kind == "mi":
                        emit(f"  const lm_f2 {p}ar = lm_add2({ar}, {bi}), {p}ai = lm_sub2({ai}, {br});")
                        emit(f"  const lm_f2 {p}br = lm_sub2({ar}, {bi}), {p}bi = lm_add2({ai}, {br});")
                        ops2 += 4
                    elif kind == "tan":
                        emit(f"  const lm_f2 {p}ur = lm_fma2(lm_bcast({lit(t)}), {bi}, {br}), "
                             f"{p}ui = lm_fma2(lm_bcast({lit(-t)}), {br}, {bi});")
                        emit(f"  const lm_f2 {p}ar = lm_fma2(lm_bcast({lit(c)}), {p}ur, {ar}), "
                             f"{p}ai = lm_fma2(lm_bcast({lit(c)}), {p}ui, {ai});")
                        emit(f"  const lm_f2 {p}br = lm_fma2(lm_bcast({lit(-c)}), {p}ur, {ar}), "
                             f"{p}bi = lm_fma2(lm_bcast({lit(-c)}), {p}ui, {ai});")
                        ops2 += 6
                    else:
                        emit(f"  const lm_f2 {p}ur = lm_fma2(lm_bcast({lit(-t)}), {bi}, {br}), "
                             f"{p}ui = lm_fma2(lm_bcast({lit(t)}), {br}, {bi});")
                        emit(f"  const lm_f2 {p}ar = lm_fma2(lm_bcast({lit(sn)}), {p}ui, {ar}), "
                             f"{p}ai = lm_fma2(lm_bcast({lit(-sn)}), {p}ur, {ai});")
                        emit(f"  const lm_f2 {p}br = lm_fma2(lm_bcast({lit(-sn)}), {p}ui, {ar}), "
                             f"{p}bi = lm_fma2(lm_bcast({lit(sn)}), {p}ur, {ai});")
                        ops2 += 6
                    cur[ia] = (f"{p}ar", f"{p}ai")
                    cur[ib] = (f"{p}br", f"{p}bi")
        # last stage: X[i] = E[i] + wn^i O[i], X[i+n/2] = E[i] - wn^i O[i]; E = lo halves, O = hi halves
        for i in range(h):
            R, I = cur[i]
            ar, ai, br, bi = f"lm_lo({R})", f"lm_lo({I})", f"lm_hi({R})", f"lm_hi({I})"
            kind, c, sn, t = twiddle_kind(i, n)
            p = f"f{i}" if count == 1 else f"f{b}_{i}"
            lo, hi = b * n + i, b * n + i + h
            if kind == "one":
                emit(f"  xr[{lo}] = {ar} + {br}; xi[{lo}] = {ai} + {bi}; xr[{hi}] = {ar} - {br}; xi[{hi}] = {ai} - {bi};")
                ops1 += 4
            elif kind == "mi":
                emit(f"  xr[{lo}] = {ar} + {bi}; xi[{lo}] = {ai} - {br}; xr[{hi}] = {ar} - {bi}; xi[{hi}] = {ai} + {br};")
                ops1 += 4
            elif kind == "tan":
                emit(f"  const float {p}ur = fmaf({lit(t)}, {bi}, {br}), {p}ui = fmaf({lit(-t)}, {br}, {bi});")
                emit(f"  xr[{lo}] = fmaf({lit(c)}, {p}ur, {ar}); xi[{lo}] = fmaf({lit(c)}, {p}ui, {ai}); "
                     f"xr[{hi}] = fmaf({lit(-c)}, {p}ur, {ar}); xi[{hi}] = fmaf({lit(-c)}, {p}ui, {ai});")
                ops1 += 6
            else:
                emit(f"  const float {p}ur = fmaf({lit(-t)}, {bi}, {br}), {p}ui = fmaf({lit(t)}, {br}, {bi});")
                emit(f"  xr[{lo}] = fmaf({lit(sn)}, {p}ui, {ar}); xi[{lo}] = fmaf({lit(-sn)}, {p}ur, {ai}); "
                     f"xr[{hi}] = fmaf({lit(-sn)}, {p}ui, {ar}); xi[{hi}] = fmaf({lit(sn)}, {p}ur, {ai});")
                ops1 += 6
    emit("}")
    emit(f"// {name}: {ops2} packed f32x2 ops + {ops1} scalar ops")
    return "\n".join(out)


def main() -> None:
    print("// GENERATED by gen_fft.py -- do not edit.  Register-resident forward FFTs.")
    print("#pragma once")
    print('#include "lm_f2.cuh"')
    for n in (8, 16, 32):
        print()
        print(gen_scalar(n))
    print()
    print(gen_aos(32))
    print()
    print(gen_aos(32, first_stage=2))
    for n in (32, 16, 8):
        print()
        print(gen_soa(n))


if __name__ == "__main__":
    main()
