// Device field library: 256-bit prime-field arithmetic on 8 x u32 limbs for BN254 / BLS12-381 Fr.
//
// GPU counterpart of the reference's Fr_* runtime (c_elements/<prime>/fr.asm,
// c_elements/generic/fr.cpp); value semantics are those of SURVEY.md Appendix C.
// Everything here is `__host__ __device__` plain C++ so that tests/ can compile the very
// same source for the CPU and check it against the oracle without a GPU; the PTX fast
// path of the Montgomery product is selected only under __CUDA_ARCH__.
#pragma once
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define CW_HD __host__ __device__ __forceinline__
#else
#define CW_HD inline
#endif

namespace cw {

typedef uint32_t u32;
typedef uint64_t u64;

struct FrParams {
    u32 q[8];     // modulus
    u32 half[8];  // q >> 1  (generic/fr.cpp:9)
    u32 r1[8];    // 2^256 mod q : Montgomery image of 1
    u32 r2[8];    // 2^512 mod q
    u32 qm2[8];   // q - 2 (Fermat exponent)
    u32 np32;     // -q^-1 mod 2^32
    u32 qbits;    // 254 / 255 / 256; 64 for goldilocks
    u32 top_mask; // lboMask on the limb of the top bit (generic/fr.cpp:16)
    u32 pad;
};

// ---- raw 256-bit helpers -----------------------------------------------------------------------
// On the device the 8-limb add / subtract are single carry chains (add.cc / addc.cc: 9 integer
// instructions instead of ~24 with 64-bit emulation); the host build keeps the portable form.
CW_HD u32 u256_add(u32 *r, const u32 *a, const u32 *b) {  // returns carry
#if defined(__CUDA_ARCH__)
    u32 r0, r1, r2, r3, r4, r5, r6, r7, c;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=&r"(r0), "=&r"(r1), "=&r"(r2), "=&r"(r3), "=&r"(r4), "=&r"(r5), "=&r"(r6), "=&r"(r7), "=&r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3; r[4] = r4; r[5] = r5; r[6] = r6; r[7] = r7;
    return c;
#else
    u64 c = 0;
    for (int i = 0; i < 8; ++i) {
        c += (u64)a[i] + b[i];
        r[i] = (u32)c;
        c >>= 32;
    }
    return (u32)c;
#endif
}
CW_HD u32 u256_sub(u32 *r, const u32 *a, const u32 *b) {  // returns borrow (0 / 1)
#if defined(__CUDA_ARCH__)
    u32 r0, r1, r2, r3, r4, r5, r6, r7, c;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(r0), "=&r"(r1), "=&r"(r2), "=&r"(r3), "=&r"(r4), "=&r"(r5), "=&r"(r6), "=&r"(r7), "=&r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3; r[4] = r4; r[5] = r5; r[6] = r6; r[7] = r7;
    return c & 1u;  // 0xFFFFFFFF when the chain ends with a borrow
#else
    u32 br = 0;
    for (int i = 0; i < 8; ++i) {
        u64 t = (u64)a[i] - b[i] - br;
        r[i] = (u32)t;
        br = (u32)(t >> 63);
    }
    return br;
#endif
}
CW_HD bool u256_geq(const u32 *a, const u32 *b) {  // a >= b
    u32 t[8];
    return u256_sub(t, a, b) == 0;
}
CW_HD bool u256_gt(const u32 *a, const u32 *b) { return !u256_geq(b, a); }
CW_HD bool u256_is_zero(const u32 *a) {
    u32 o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a[i];
    return o == 0;
}
CW_HD bool u256_eq(const u32 *a, const u32 *b) {
    u32 o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a[i] ^ b[i];
    return o == 0;
}
CW_HD void u256_set(u32 *r, const u32 *a) {
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = a[i];
}
CW_HD void u256_set_u32(u32 *r, u32 v) {
    r[0] = v;
#pragma unroll
    for (int i = 1; i < 8; ++i) r[i] = 0;
}
// r = r >= q ? r - q : r
CW_HD void fr_cond_sub(u32 *r, const FrParams &P) {
    u32 t[8];
    u32 br = u256_sub(t, r, P.q);
    if (!br) u256_set(r, t);
}

// ---- add / sub / neg (generic/fr.cpp:19-86) ----------------------------------------------------
CW_HD void fr_add(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 s[8], t[8];
    u32 c = u256_add(s, a, b);
    u32 br = u256_sub(t, s, P.q);
    bool use_t = c || !br;
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = use_t ? t[i] : s[i];
}
CW_HD void fr_sub(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 s[8], t[8];
    u32 br = u256_sub(s, a, b);
    u256_add(t, s, P.q);
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = br ? t[i] : s[i];
}
CW_HD void fr_neg(u32 *r, const u32 *a, const FrParams &P) {
    u32 t[8];
    u256_sub(t, P.q, a);
    bool z = u256_is_zero(a);
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = z ? 0u : t[i];
}

// ---- Montgomery product a*b*2^-256 mod q, CIOS (generic/fr.cpp:110-164; bn128/fr.asm:365-531) --
CW_HD void fr_mont_mul_c(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 t[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        u64 c = 0;
        u32 bi = b[i];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            c += (u64)a[j] * bi + t[j];
            t[j] = (u32)c;
            c >>= 32;
        }
        c += t[8];
        t[8] = (u32)c;
        u32 t9 = (u32)(c >> 32);
        u32 m = t[0] * P.np32;
        c = (u64)m * P.q[0] + t[0];
        c >>= 32;
#pragma unroll
        for (int j = 1; j < 8; ++j) {
            c += (u64)m * P.q[j] + t[j];
            t[j - 1] = (u32)c;
            c >>= 32;
        }
        c += t[8];
        t[7] = (u32)c;
        t[8] = t9 + (u32)(c >> 32);
    }
    // the CIOS result is < 2q: for the 254 / 255-bit moduli it fits 256 bits (t[8] == 0); for a 256-bit modulus
    // (secq256r1) the ninth limb can be 1, and then the subtraction is due whatever its borrow says
    u32 d[8];
    u32 br = u256_sub(d, t, P.q);
    const bool sub = t[8] != 0u || !br;
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = sub ? d[i] : t[i];
}

#if defined(__CUDA_ARCH__)
// PTX carry-chain CIOS on the integer (IMAD) pipe: per outer iteration the 8 low halves and the 8 high
// halves of a*b[i] are accumulated as two pure carry chains (mad.lo.cc / madc.lo.cc, mad.hi.cc /
// madc.hi.cc), likewise for m*q, then the accumulator moves down one limb.  39 integer instructions per
// iteration, 8 iterations, one conditional subtraction.  Same result as fr_mont_mul_c.  MEASURED SLOWER on
// B200 than the portable form, which nvcc compiles to IMAD.WIDE (both halves of a limb product in one
// instruction): 43.4 vs 49.5 G modmul/s (scripts/mul_bench.py) - kept behind -DCW_MONT_PTX for reference.
__device__ __forceinline__ void fr_mont_step(u32 *t, const u32 *a, u32 bi, const FrParams &P) {
    u32 m;
    asm("{\n\t"
        "mad.lo.cc.u32   %0, %11, %19, %0;\n\t"
        "madc.lo.cc.u32  %1, %12, %19, %1;\n\t"
        "madc.lo.cc.u32  %2, %13, %19, %2;\n\t"
        "madc.lo.cc.u32  %3, %14, %19, %3;\n\t"
        "madc.lo.cc.u32  %4, %15, %19, %4;\n\t"
        "madc.lo.cc.u32  %5, %16, %19, %5;\n\t"
        "madc.lo.cc.u32  %6, %17, %19, %6;\n\t"
        "madc.lo.cc.u32  %7, %18, %19, %7;\n\t"
        "addc.cc.u32     %8, %8, 0;\n\t"
        "addc.u32        %9, 0, 0;\n\t"
        "mad.hi.cc.u32   %1, %11, %19, %1;\n\t"
        "madc.hi.cc.u32  %2, %12, %19, %2;\n\t"
        "madc.hi.cc.u32  %3, %13, %19, %3;\n\t"
        "madc.hi.cc.u32  %4, %14, %19, %4;\n\t"
        "madc.hi.cc.u32  %5, %15, %19, %5;\n\t"
        "madc.hi.cc.u32  %6, %16, %19, %6;\n\t"
        "madc.hi.cc.u32  %7, %17, %19, %7;\n\t"
        "madc.hi.cc.u32  %8, %18, %19, %8;\n\t"
        "addc.u32        %9, %9, 0;\n\t"
        "mul.lo.u32      %10, %0, %28;\n\t"
        "mad.lo.cc.u32   %0, %10, %20, %0;\n\t"
        "madc.lo.cc.u32  %1, %10, %21, %1;\n\t"
        "madc.lo.cc.u32  %2, %10, %22, %2;\n\t"
        "madc.lo.cc.u32  %3, %10, %23, %3;\n\t"
        "madc.lo.cc.u32  %4, %10, %24, %4;\n\t"
        "madc.lo.cc.u32  %5, %10, %25, %5;\n\t"
        "madc.lo.cc.u32  %6, %10, %26, %6;\n\t"
        "madc.lo.cc.u32  %7, %10, %27, %7;\n\t"
        "addc.cc.u32     %8, %8, 0;\n\t"
        "addc.u32        %9, %9, 0;\n\t"
        "mad.hi.cc.u32   %1, %10, %20, %1;\n\t"
        "madc.hi.cc.u32  %2, %10, %21, %2;\n\t"
        "madc.hi.cc.u32  %3, %10, %22, %3;\n\t"
        "madc.hi.cc.u32  %4, %10, %23, %4;\n\t"
        "madc.hi.cc.u32  %5, %10, %24, %5;\n\t"
        "madc.hi.cc.u32  %6, %10, %25, %6;\n\t"
        "madc.hi.cc.u32  %7, %10, %26, %7;\n\t"
        "madc.hi.cc.u32  %8, %10, %27, %8;\n\t"
        "addc.u32        %9, %9, 0;\n\t"
        "}"
        : "+r"(t[0]), "+r"(t[1]), "+r"(t[2]), "+r"(t[3]), "+r"(t[4]), "+r"(t[5]), "+r"(t[6]), "+r"(t[7]), "+r"(t[8]),
          "+r"(t[9]), "=&r"(m)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(bi),
          "r"(P.q[0]), "r"(P.q[1]), "r"(P.q[2]), "r"(P.q[3]), "r"(P.q[4]), "r"(P.q[5]), "r"(P.q[6]), "r"(P.q[7]),
          "r"(P.np32));
    // t[0] is now zero: move the accumulator down one limb
#pragma unroll
    for (int j = 0; j < 9; ++j) t[j] = t[j + 1];
    t[9] = 0;
}
__device__ __forceinline__ void fr_mont_mul_ptx(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 t[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) fr_mont_step(t, a, b[i], P);
    u32 d[8];
    u32 br = u256_sub(d, t, P.q);  // result < 2q; t[8] is 0 unless the modulus has 256 bits
    const bool sub = t[8] != 0u || !br;
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = sub ? d[i] : t[i];
}
#endif

CW_HD void fr_mont_mul(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
#if defined(__CUDA_ARCH__) && defined(CW_MONT_PTX)
    fr_mont_mul_ptx(r, a, b, P);
#else
    fr_mont_mul_c(r, a, b, P);
#endif
}

CW_HD void fr_to_mont(u32 *r, const u32 *a, const FrParams &P) { fr_mont_mul(r, a, P.r2, P); }
CW_HD void fr_from_mont(u32 *r, const u32 *a, const FrParams &P) {
    u32 one[8];
    u256_set_u32(one, 1);
    fr_mont_mul(r, a, one, P);
}

// ---- exponentiation in the Montgomery domain: base = xR, exponent canonical -> x^e R -------------
// Fr_pow (generic/fr.cpp:2877-2893) / Fr_inv via Fermat (x^(q-2); 0 -> 0 like the pinned
// behaviour of mpz_invert's ignored failure, generic/fr.cpp:2895-2906).
CW_HD void fr_pow_mont(u32 *r, const u32 *base, const u32 *e_in, const FrParams &P) {
    // left-to-right square-and-multiply; the exponent is consumed by shifting a register copy so
    // that no array is indexed dynamically (dynamic indexing would push it to local memory)
    u32 acc[8], e[8];
    u256_set(acc, P.r1);
    u256_set(e, e_in);
    bool started = false;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 0; i < 256; ++i) {
        u32 bit = e[7] >> 31;
#pragma unroll
        for (int j = 7; j > 0; --j) e[j] = (e[j] << 1) | (e[j - 1] >> 31);
        e[0] <<= 1;
        if (started) {
            u32 t[8];
            fr_mont_mul(t, acc, acc, P);
            u256_set(acc, t);
        }
        if (bit) {
            if (started) {
                u32 t[8];
                fr_mont_mul(t, acc, base, P);
                u256_set(acc, t);
            } else {
                u256_set(acc, base);
                started = true;
            }
        }
    }
    u256_set(r, acc);
}
CW_HD void fr_inv_mont_fermat(u32 *r, const u32 *a, const FrParams &P) { fr_pow_mont(r, a, P.qm2, P); }   // a^(q-2): ~380 products

// ---- modular inverse by division steps ("safegcd", Bernstein - Yang 2019, in the form of libsecp256k1's modinv32) ----
// The reference inverts with GMP's mpz_invert (generic/fr.cpp:2895-2906).  Fermat's ladder costs ~380 Montgomery products per
// inverse; 600 division steps on (f, g) = (q, x) cost 20 rounds of 30 branch-free single-word steps that produce a 2x2
// transition matrix, applied to the full-size (f, g) and to the Bezout pair (d, e) mod q - about a tenth of the work, and
// no step depends on the data (a warp of 32 instances stays converged).  Numbers are 9 signed limbs of 30 bits.
// x = 0 gives 0, as the reference's result on 0 (SURVEY Appendix D).
struct Inv30 {
    int32_t v[9];
};
CW_HD void inv30_from_u256(Inv30 &r, const u32 *a) {
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        const int bit = 30 * i, w = bit >> 5, sh = bit & 31;
        u64 x = (u64)a[w] >> sh;
        if (sh > 2 && w + 1 < 8) x |= (u64)a[w + 1] << (32 - sh);
        r.v[i] = (int32_t)((u32)x & 0x3FFFFFFFu);
    }
}
CW_HD void inv30_to_u256(u32 *a, const Inv30 &r) {   // limbs in [0, 2^30), value < 2^256
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        const int bit = 30 * i, w = bit >> 5, sh = bit & 31;
        const u64 x = (u64)(u32)r.v[i] << sh;
        a[w] |= (u32)x;
        if (w + 1 < 8) a[w + 1] |= (u32)(x >> 32);
    }
}
// 30 division steps on the low words of f (odd) and g; the transition matrix t = {u, v, q, r} satisfies
// 2^30 * (f', g') = t * (f, g).  zeta = -(delta + 1/2).
CW_HD int32_t inv30_divsteps(int32_t zeta, u32 f0, u32 g0, int32_t *t) {
    u32 u = 1, v = 0, q = 0, r = 1, f = f0, g = g0;
#pragma unroll 6
    for (int i = 0; i < 30; ++i) {
        u32 mask1 = (u32)(zeta >> 31);           // zeta < 0
        const u32 mask2 = 0u - (g & 1u);         // g odd
        const u32 x = (f ^ mask1) - mask1, y = (u ^ mask1) - mask1, z = (v ^ mask1) - mask1;
        g += x & mask2;
        q += y & mask2;
        r += z & mask2;
        mask1 &= mask2;
        zeta = (int32_t)(((u32)zeta ^ mask1) - 1u);
        f += g & mask1;
        u += q & mask1;
        v += r & mask1;
        g >>= 1;
        u <<= 1;
        v <<= 1;
    }
    t[0] = (int32_t)u; t[1] = (int32_t)v; t[2] = (int32_t)q; t[3] = (int32_t)r;
    return zeta;
}
// (f, g) <- t * (f, g) / 2^30 (exact)
CW_HD void inv30_update_fg(Inv30 &f, Inv30 &g, const int32_t *t) {
    const int64_t u = t[0], v = t[1], q = t[2], r = t[3];
    int64_t cf = u * f.v[0] + v * g.v[0], cg = q * f.v[0] + r * g.v[0];
    cf >>= 30;
    cg >>= 30;
#pragma unroll
    for (int i = 1; i < 9; ++i) {
        const int64_t fi = f.v[i], gi = g.v[i];
        cf += u * fi + v * gi;
        cg += q * fi + r * gi;
        f.v[i - 1] = (int32_t)((u32)cf & 0x3FFFFFFFu);
        g.v[i - 1] = (int32_t)((u32)cg & 0x3FFFFFFFu);
        cf >>= 30;
        cg >>= 30;
    }
    f.v[8] = (int32_t)cf;
    g.v[8] = (int32_t)cg;
}
// (d, e) <- t * (d, e) / 2^30 mod m, with d, e kept in (-2m, m); minv30 = m^-1 mod 2^30
CW_HD void inv30_update_de(Inv30 &d, Inv30 &e, const int32_t *t, const Inv30 &m, u32 minv30) {
    const int32_t u = t[0], v = t[1], q = t[2], r = t[3];
    const int32_t sd = d.v[8] >> 31, se = e.v[8] >> 31;
    int32_t md = (u & sd) + (v & se), me = (q & sd) + (r & se);
    int64_t cd = (int64_t)u * d.v[0] + (int64_t)v * e.v[0], ce = (int64_t)q * d.v[0] + (int64_t)r * e.v[0];
    // multiples of the modulus that clear the low 30 bits
    md -= (int32_t)((minv30 * (u32)cd + (u32)md) & 0x3FFFFFFFu);
    me -= (int32_t)((minv30 * (u32)ce + (u32)me) & 0x3FFFFFFFu);
    cd += (int64_t)m.v[0] * md;
    ce += (int64_t)m.v[0] * me;
    cd >>= 30;
    ce >>= 30;
#pragma unroll
    for (int i = 1; i < 9; ++i) {
        cd += (int64_t)u * d.v[i] + (int64_t)v * e.v[i] + (int64_t)m.v[i] * md;
        ce += (int64_t)q * d.v[i] + (int64_t)r * e.v[i] + (int64_t)m.v[i] * me;
        d.v[i - 1] = (int32_t)((u32)cd & 0x3FFFFFFFu);
        e.v[i - 1] = (int32_t)((u32)ce & 0x3FFFFFFFu);
        cd >>= 30;
        ce >>= 30;
    }
    d.v[8] = (int32_t)cd;
    e.v[8] = (int32_t)ce;
}
// r in (-2m, m), negated when sign < 0, brought to [0, m)
CW_HD void inv30_normalize(Inv30 &r, int32_t sign, const Inv30 &m) {
    int32_t cond_add = r.v[8] >> 31;
    const int32_t cond_neg = sign >> 31;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        r.v[i] += m.v[i] & cond_add;
        r.v[i] = (r.v[i] ^ cond_neg) - cond_neg;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        r.v[i + 1] += r.v[i] >> 30;
        r.v[i] &= 0x3FFFFFFF;
    }
    cond_add = r.v[8] >> 31;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.v[i] += m.v[i] & cond_add;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        r.v[i + 1] += r.v[i] >> 30;
        r.v[i] &= 0x3FFFFFFF;
    }
}
// canonical x < q  ->  x^-1 mod q (canonical), 0 -> 0.  (Five 9-limb numbers: inlined into the interpreter's hot loop it
// cost 16 % of the headline throughput in spills - the interpreter runs INV / POW in a pass of their own, kernels.cuh.)
CW_HD void fr_modinv(u32 *out, const u32 *x, const FrParams &P) {
    Inv30 m, f, g, d, e;
    inv30_from_u256(m, P.q);
    f = m;
    inv30_from_u256(g, x);
#pragma unroll
    for (int i = 0; i < 9; ++i) { d.v[i] = 0; e.v[i] = 0; }
    e.v[0] = 1;
    const u32 minv30 = (0u - P.np32) & 0x3FFFFFFFu;   // np32 = -q^-1 mod 2^32
    int32_t zeta = -1;
#pragma unroll 1
    for (int it = 0; it < 20; ++it) {       // 600 >= 590 division steps: enough for 256-bit inputs
        int32_t t[4];
        zeta = inv30_divsteps(zeta, (u32)f.v[0] | ((u32)f.v[1] << 30), (u32)g.v[0] | ((u32)g.v[1] << 30), t);
        inv30_update_de(d, e, t, m, minv30);
        inv30_update_fg(f, g, t);
    }
    // g = 0, f = +-gcd(x, q) = +-1 (or +-q for x = 0, where d = 0): d * sign(f) is the inverse
    inv30_normalize(d, f.v[8], m);
    inv30_to_u256(out, d);
}
// a = x R  ->  x^-1 R:  modinv gives x^-1 R^-1, two products with R^2 restore the factor
CW_HD void fr_inv_mont(u32 *r, const u32 *a, const FrParams &P) {
#ifdef CW_INV_FERMAT   // (A/B builds: scripts/inv_bench.py)
    fr_inv_mont_fermat(r, a, P);
#else
    u32 t[8], s[8];
    fr_modinv(t, a, P);
    fr_mont_mul(s, t, P.r2, P);
    fr_mont_mul(r, s, P.r2, P);
#endif
}

// ---- shifts on the canonical integer (generic/fr.cpp:329-364,1995-2027,2157-2307) ----------------
// barrel shifters with static register indices only
CW_HD void u256_shl(u32 *r, const u32 *a, u32 k) {  // 0 <= k < 256, result mod 2^256
    u32 t[8];
    u256_set(t, a);
    if (k & 128) {
#pragma unroll
        for (int i = 7; i >= 0; --i) t[i] = i >= 4 ? t[i - 4] : 0;
    }
    if (k & 64) {
#pragma unroll
        for (int i = 7; i >= 0; --i) t[i] = i >= 2 ? t[i - 2] : 0;
    }
    if (k & 32) {
#pragma unroll
        for (int i = 7; i >= 0; --i) t[i] = i >= 1 ? t[i - 1] : 0;
    }
    u32 s = k & 31;
    if (s) {
#pragma unroll
        for (int i = 7; i > 0; --i) t[i] = (t[i] << s) | (t[i - 1] >> (32 - s));
        t[0] <<= s;
    }
    u256_set(r, t);
}
CW_HD void u256_shr(u32 *r, const u32 *a, u32 k) {
    u32 t[8];
    u256_set(t, a);
    if (k & 128) {
#pragma unroll
        for (int i = 0; i < 8; ++i) t[i] = i + 4 < 8 ? t[i + 4] : 0;
    }
    if (k & 64) {
#pragma unroll
        for (int i = 0; i < 8; ++i) t[i] = i + 2 < 8 ? t[i + 2] : 0;
    }
    if (k & 32) {
#pragma unroll
        for (int i = 0; i < 8; ++i) t[i] = i + 1 < 8 ? t[i + 1] : 0;
    }
    u32 s = k & 31;
    if (s) {
#pragma unroll
        for (int i = 0; i < 7; ++i) t[i] = (t[i] >> s) | (t[i + 1] << (32 - s));
        t[7] >>= s;
    }
    u256_set(r, t);
}
CW_HD void fr_mask_wrap(u32 *r, const FrParams &P) {  // top-limb mask then one conditional subtraction
    if (P.qbits > 224u) r[7] &= P.top_mask;   // every 256-bit prime
    else {                                    // goldilocks (c_elements/goldilocks/fr.hpp:177-181,255-270): 64-bit words
        const u32 top = (P.qbits - 1u) >> 5;
#pragma unroll
        for (int i = 0; i < 8; ++i) r[i] = (u32)i < top ? r[i] : ((u32)i == top ? (r[i] & P.top_mask) : 0u);
    }
    fr_cond_sub(r, P);
}
// decode the shift amount: returns 0 = plain by k, 1 = opposite direction by k, 2 = result is zero
CW_HD int fr_shift_kind(const u32 *b, u32 &k, const FrParams &P) {
    u32 hi = b[1] | b[2] | b[3] | b[4] | b[5] | b[6] | b[7];
    if (!hi && b[0] < P.qbits) { k = b[0]; return 0; }
    u32 nb[8];
    u256_sub(nb, P.q, b);  // "negative" amount -j is stored as q-j
    hi = nb[1] | nb[2] | nb[3] | nb[4] | nb[5] | nb[6] | nb[7];
    if (!hi && nb[0] < P.qbits) { k = nb[0]; return 1; }
    k = 0;
    return 2;
}
CW_HD void fr_shl(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 k;
    int kind = fr_shift_kind(b, k, P);
    if (kind == 0) { u256_shl(r, a, k); fr_mask_wrap(r, P); }
    else if (kind == 1) u256_shr(r, a, k);
    else u256_set_u32(r, 0);
}
CW_HD void fr_shr(u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 k;
    int kind = fr_shift_kind(b, k, P);
    if (kind == 0) u256_shr(r, a, k);
    else if (kind == 1) { u256_shl(r, a, k); fr_mask_wrap(r, P); }
    else u256_set_u32(r, 0);
}

// ---- comparisons on val(x) = x > half ? x - q : x (generic/fr.cpp:1184-1218,1294-1363) ----------
CW_HD bool fr_lt(const u32 *a, const u32 *b, const FrParams &P) {
    bool an = u256_gt(a, P.half), bn = u256_gt(b, P.half);
    if (an != bn) return an;
    return u256_gt(b, a);
}

// ---- integer division of canonical values (Fr_idiv / Fr_mod, generic/fr.cpp:2835-2875) ----------
// returns false on division by zero (the reference process aborts inside GMP)
CW_HD u32 u256_clz(const u32 *a) {  // leading zero bits, 256 for zero
    u32 n = 0;
    bool done = false;
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        if (!done) {
            if (a[i]) {
                u32 x = a[i], c = 0;
                while (!(x & 0x80000000u)) { x <<= 1; ++c; }
                n += c;
                done = true;
            } else n += 32;
        }
    }
    return n;
}
CW_HD bool u256_divmod(u32 *quo, u32 *rem, const u32 *a, const u32 *b) {
    if (u256_is_zero(b)) {
        u256_set_u32(quo, 0);
        u256_set_u32(rem, 0);
        return false;
    }
    // power-of-two divisor: shift / mask
    u32 lzb = u256_clz(b);
    {
        u32 single[8], one[8];
        u256_set_u32(one, 1);
        u256_shl(single, one, 255 - lzb);
        if (u256_eq(single, b)) {
            u32 bit = 255 - lzb;
            u256_shr(quo, a, bit);
            u32 t[8];
            u256_shl(t, quo, bit);
            u256_sub(rem, a, t);
            return true;
        }
    }
    // restoring division, one bit per step; the numerator is consumed from a shifting register copy
    u32 lza = u256_clz(a);
    u32 n[8], q[8], r[8];
    if (lza == 256) {
        u256_set_u32(quo, 0);
        u256_set_u32(rem, 0);
        return true;
    }
    u256_shl(n, a, lza);
    u256_set_u32(q, 0);
    u256_set_u32(r, 0);
    int steps = 256 - (int)lza;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 0; i < steps; ++i) {
        u32 carry = n[7] >> 31;
#pragma unroll
        for (int j = 7; j > 0; --j) n[j] = (n[j] << 1) | (n[j - 1] >> 31);
        n[0] <<= 1;
        const u32 rtop = r[7] >> 31;  // r < b: with a 256-bit divisor 2r + carry can leave 256 bits - then it exceeds b for sure
#pragma unroll
        for (int j = 7; j > 0; --j) r[j] = (r[j] << 1) | (r[j - 1] >> 31);
        r[0] = (r[0] << 1) | carry;
        u32 t[8];
        u32 br = u256_sub(t, r, b);   // (mod 2^256: the right difference also when the shift overflowed)
#pragma unroll
        for (int j = 7; j > 0; --j) q[j] = (q[j] << 1) | (q[j - 1] >> 31);
        q[0] <<= 1;
        if (rtop || !br) {
            u256_set(r, t);
            q[0] |= 1;
        }
    }
    u256_set(quo, q);
    u256_set(rem, r);
    return true;
}

// ---- one tape instruction ----------------------------------------------------------------------
// Opcodes are cw_op (include/circom_b200.h).  Operands arrive in the representation the lowering
// chose (flatten.cpp); `err` is set to 1 on division by zero (host builds: also on a typed operator whose range
// claim fails, below).  Returns true if r holds a result.
enum {
    OP_MUL = 1, OP_ADD = 3, OP_SUB = 4, OP_POW = 5, OP_IDIV = 6, OP_MOD = 7, OP_SHL = 8, OP_SHR = 9,
    OP_LEQ = 10, OP_GEQ = 11, OP_LT = 12, OP_GT = 13, OP_EQ = 14, OP_NEQ = 15, OP_LOR = 16, OP_LAND = 17,
    OP_LNOT = 18, OP_BOR = 19, OP_BAND = 20, OP_BXOR = 21, OP_BNOT = 22, OP_NEG = 23, OP_COPY = 24,
    OP_SELECT = 25, OP_ASSERT = 26, OP_ASSERT_EQ = 27, OP_INV = 28,
    OP_BITS = 29,         // (a >> k) & (2^m - 1), imm = k | m << 16  (fused `(x >> k) & mask` hints)
    OP_ASSERT_BOOL = 30,  // a == 0 || a == b  (b = the constant one in a's representation)
    OP_MULSMALL = 31,     // a * b as integers, statically known to stay below q (no reduction)
    OP_BITSIP = 32,       // a & ((2^len - 1) << lo), imm = lo | len << 8  (sum of adjacent bit fields)
    OP_ASSERT_FITS = 33,  // a < 2^m, m = b[0]  (recomposition check of a bit decomposition)
    // width-typed operators: the lowering's range analysis proves the canonical result narrow, so the integer result
    // is the field result and only the limbs that can be non-zero are computed.  (Below FOP_JMP: OP_CALL must stay the
    // largest opcode of a level.)
    OP_ADD_NR = 34,        // a + b < q: no modular correction
    OP_ADD128 = 35,        // a + b < 2^128: a 4-limb addition
    OP_MULSMALL128 = 36,   // a * b < 2^128 as integers: the low 4 limbs of the product
    OP_MULSMALL192 = 37,   // a * b < 2^192 as integers: the low 6 limbs
    OP_SHRI = 38,          // a >> b, b a constant below qbits (no decoding of the amount against q)
    OP_SHLI = 39           // a << b, b a constant below qbits, the result proved below q (no reduction)
};

// low 256 bits of the integer product (36 limb products instead of CIOS' 128)
CW_HD void u256_mul_lo(u32 *r, const u32 *a, const u32 *b) {
    u32 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        u64 c = 0;
#pragma unroll
        for (int j = 0; j + i < 8; ++j) {
            c += (u64)a[j] * b[i] + t[i + j];
            t[i + j] = (u32)c;
            c >>= 32;
        }
    }
    u256_set(r, t);
}
// low K limbs of the integer product, the limbs above them zero (K (K + 1) / 2 limb products)
template <int K>
CW_HD void u256_mul_lo_k(u32 *r, const u32 *a, const u32 *b) {
    u32 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = 0;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        u64 c = 0;
#pragma unroll
        for (int j = 0; j + i < K; ++j) {
            c += (u64)a[j] * b[i] + t[i + j];
            t[i + j] = (u32)c;
            c >>= 32;
        }
    }
    u256_set(r, t);
}
CW_HD void u256_add_lo4(u32 *r, const u32 *a, const u32 *b) {   // a + b < 2^128
    u64 c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        c += (u64)a[i] + b[i];
        r[i] = (u32)c;
        c >>= 32;
    }
#pragma unroll
    for (int i = 4; i < 8; ++i) r[i] = 0;
}
CW_HD void u256_bits(u32 *r, const u32 *a, u32 imm) {
    u32 k = imm & 0xFFFFu, m = (imm >> 16) & 0xFFu;
    u32 t[8];
    u256_shr(t, a, k);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int lo = i * 32;
        u32 mask = (int)m >= lo + 32 ? 0xFFFFFFFFu : ((int)m <= lo ? 0u : ((1u << (m - lo)) - 1u));
        r[i] = t[i] & mask;
    }
}

CW_HD void u256_bits_in_place(u32 *r, const u32 *a, u32 imm) {
    u32 lo = imm & 0xFFu, len = imm >> 8, hi = lo + len;  // keep bits [lo, hi)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        u32 b0 = 32u * i, b1 = b0 + 32u;
        u32 m = 0;
        if (hi > b0 && lo < b1) {
            u32 from = lo > b0 ? lo - b0 : 0u, to = hi < b1 ? hi - b0 : 32u;  // bit range inside this limb
            u32 w = to - from;
            m = (w >= 32u ? 0xFFFFFFFFu : ((1u << w) - 1u)) << from;
        }
        r[i] = a[i] & m;
    }
}
CW_HD u32 u256_bitlen(const u32 *a) {
    u32 n = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (a[i]) {
            u32 x = a[i], c = 0;
            while (x) { x >>= 1; ++c; }
            n = 32u * i + c;
        }
    }
    return n;
}

// a width-typed operator's result r equals the generic operator's, and is below q
CW_HD bool fr_typed_holds(u32 opcode, const u32 *r, const u32 *a, const u32 *b, const FrParams &P) {
    u32 g[8];
    if (opcode == OP_ADD_NR || opcode == OP_ADD128) fr_add(g, a, b, P);
    else if (opcode == OP_MULSMALL128 || opcode == OP_MULSMALL192) u256_mul_lo(g, a, b);
    else if (opcode == OP_SHRI) fr_shr(g, a, b, P);
    else fr_shl(g, a, b, P);
    return u256_eq(g, r) && !u256_geq(r, P.q);
}

// SLOW = false leaves out the two operators that are loops of hundreds of steps (INV, POW): the interpreter runs them
// in a pass of their own so that their code and registers stay out of its hot loop (kernels.cuh)
template <bool SLOW>
CW_HD void fr_exec_t(u32 opcode, u32 *r, const u32 *a, const u32 *b, u32 imm, const FrParams &P, int &err) {
    switch (opcode) {
        case OP_BITSIP: u256_bits_in_place(r, a, imm); break;
        case OP_BITS: u256_bits(r, a, imm); break;
        case OP_MULSMALL: u256_mul_lo(r, a, b); break;
        case OP_MULSMALL128: u256_mul_lo_k<4>(r, a, b); break;
        case OP_MULSMALL192: u256_mul_lo_k<6>(r, a, b); break;
        case OP_MUL: fr_mont_mul(r, a, b, P); break;
        case OP_ADD: fr_add(r, a, b, P); break;
        case OP_ADD_NR: u256_add(r, a, b); break;
        case OP_ADD128: u256_add_lo4(r, a, b); break;
        case OP_SHRI: u256_shr(r, a, b[0]); break;
        case OP_SHLI: u256_shl(r, a, b[0]); break;
        case OP_SUB: fr_sub(r, a, b, P); break;
        case OP_NEG: fr_neg(r, a, P); break;
        case OP_INV: if (SLOW) fr_inv_mont(r, a, P); break;
        case OP_POW: if (SLOW) fr_pow_mont(r, a, b, P); break;
        case OP_IDIV: { u32 rem[8]; if (!u256_divmod(r, rem, a, b)) err = 1; break; }
        case OP_MOD: { u32 quo[8]; if (!u256_divmod(quo, r, a, b)) err = 1; break; }
        case OP_SHL: fr_shl(r, a, b, P); break;
        case OP_SHR: fr_shr(r, a, b, P); break;
        case OP_LT: u256_set_u32(r, fr_lt(a, b, P)); break;
        case OP_GT: u256_set_u32(r, fr_lt(b, a, P)); break;
        case OP_LEQ: u256_set_u32(r, !fr_lt(b, a, P)); break;
        case OP_GEQ: u256_set_u32(r, !fr_lt(a, b, P)); break;
        case OP_EQ: u256_set_u32(r, u256_eq(a, b)); break;
        case OP_NEQ: u256_set_u32(r, !u256_eq(a, b)); break;
        case OP_LOR: u256_set_u32(r, !u256_is_zero(a) || !u256_is_zero(b)); break;
        case OP_LAND: u256_set_u32(r, !u256_is_zero(a) && !u256_is_zero(b)); break;
        case OP_LNOT: u256_set_u32(r, u256_is_zero(a)); break;
        case OP_BOR:
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = a[i] | b[i];
            fr_mask_wrap(r, P);
            break;
        case OP_BAND:
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = a[i] & b[i];
            fr_mask_wrap(r, P);
            break;
        case OP_BXOR:
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = a[i] ^ b[i];
            fr_mask_wrap(r, P);
            break;
        case OP_BNOT:
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = ~a[i];
            fr_mask_wrap(r, P);
            break;
        case OP_COPY: u256_set(r, a); break;
        default: u256_set_u32(r, 0); break;
    }
#if !defined(__CUDA_ARCH__)
    // host builds (the simulator the CPU tests run tapes on): a typed operator also checks the claim of the range
    // analysis it rests on; a violation is reported like a division by zero, as an error of the instance
    if (opcode >= OP_ADD_NR && opcode <= OP_SHLI && !fr_typed_holds(opcode, r, a, b, P)) err = 1;
#endif
}
CW_HD void fr_exec(u32 opcode, u32 *r, const u32 *a, const u32 *b, u32 imm, const FrParams &P, int &err) {
    fr_exec_t<true>(opcode, r, a, b, imm, P, err);
}

// ---- canonical-in / canonical-out application of one IR operator ---------------------------------------
// (function bodies keep their variables canonical: a run-time loop cannot have its representations
// inferred statically)
CW_HD void fr_apply_canonical(u32 op, u32 *r, const u32 *a, const u32 *b, const u32 *c, const FrParams &P, int &err) {
    if (op == OP_MUL) {
        // limb arithmetic inside hint functions multiplies small values: when the integer product provably stays
        // below 2^(qbits-1) < q it IS the field product (36 limb products instead of two Montgomery products)
        if (u256_bitlen(a) + u256_bitlen(b) < P.qbits) {
            u256_mul_lo(r, a, b);
        } else {
            u32 am[8];
            fr_to_mont(am, a, P);
            fr_mont_mul(r, am, b, P);
        }
    } else if (op == 2 /* DIV */) {
        u32 bm[8], im[8];
        fr_to_mont(bm, b, P);
        fr_inv_mont(im, bm, P);
        fr_mont_mul(r, im, a, P);
    } else if (op == OP_POW) {
        u32 am[8], rm[8];
        fr_to_mont(am, a, P);
        fr_pow_mont(rm, am, b, P);
        fr_from_mont(r, rm, P);
    } else if (op == OP_SELECT) {
        bool t = !u256_is_zero(c);
        for (int k = 0; k < 8; ++k) r[k] = t ? a[k] : b[k];
    } else {
        fr_exec(op, r, a, b, 0, P, err);
    }
}

// ---- function bodies: a small register machine run by ONE thread per call --------------------------------
// circom `function`s (FunctionCodeInfo, compiler/src/circuit_design/function.rs:91-126) carry the
// data-dependent loops and branches of `<--` hints (LoopBucket / BranchBucket on Fr_isTrue,
// loop_bucket.rs:76-91, branch_bucket.rs:100-122) and index `var` arrays with run-time values
// (Fr_toInt, compute_bucket.rs:361-363).  They cannot be unrolled into the tape; a call is one tape op
// whose thread interprets the body over private registers.  Instruction = 5 words {op, d, a, b, c};
// operand: bit31 = constant-table index, bit30 = immediate, else register index.
enum { FOP_JMP = 40, FOP_JZ = 41, FOP_RET = 42, FOP_LOADX = 43, FOP_STOREX = 44, OP_CALL = 45 };
enum { VM_MAX_REGS = 192, VM_MAX_STEPS = 1 << 22, VM_MAX_DEPTH = 8 };
struct FnInfo {
    u32 code_off, n_instr, n_regs, n_params;
};
CW_HD FnInfo vm_fn(const u32 *fn_info, u32 f) {
    FnInfo fi;
    fi.code_off = fn_info[4 * (size_t)f];
    fi.n_instr = fn_info[4 * (size_t)f + 1];
    fi.n_regs = fn_info[4 * (size_t)f + 2];
    fi.n_params = fn_info[4 * (size_t)f + 3];
    return fi;
}
// A function may call functions with a smaller index (`CALL` inside a body: {45, d, function, first argument register,
// result count}; the callee's parameters are the caller's registers b .. b + n_params - 1, as the C++ producer fills
// `lvarcall`, call_bucket.rs:466-533).  Frames are stacked in the one register array of the call: the callee's frame
// starts behind the caller's.  The lowering checked at load time that the deepest chain of calls needs at most
// VM_MAX_REGS registers and VM_MAX_DEPTH frames (callee index < caller index: no recursion), so nothing is checked here.
struct VmFrame {
    u32 fn, pc, base, dst, want;
};

CW_HD void vm_operand(u32 *v, u32 o, const u32 *regs, const u32 *consts32) {
    if (o & 0x80000000u) {
        const u32 *p = consts32 + 8 * (size_t)(o & 0x3FFFFFFFu);
        for (int k = 0; k < 8; ++k) v[k] = p[k];
    } else if (o & 0x40000000u) {
        u256_set_u32(v, o & 0x3FFFFFFFu);
    } else {
        const u32 *p = regs + 8 * (size_t)o;
        for (int k = 0; k < 8; ++k) v[k] = p[k];
    }
}
// index operand -> int through the signed view (Fr_toInt, generic/fr.cpp:1146); -1 if out of range.  `limit`: the end of
// the array behind `base` (the lowering checked limit <= n_regs; without a declared extent it is n_regs)
CW_HD int vm_index(const u32 *v, u32 base, u32 limit) {
    u32 hi = v[1] | v[2] | v[3] | v[4] | v[5] | v[6] | v[7];
    if (hi || (u64)v[0] + base >= limit) return -1;
    return (int)(v[0] + base);
}
// regs: n_regs * 8 words, parameters already stored in registers 0..n_params-1.  err: 1 division by zero,
// 2 bad index / runaway loop.  `result` is the (first) returned value; a `RET` with a count c > 1 returns the c
// consecutive registers ret_base .. ret_base + c - 1 (`return arr;`, return_bucket.rs:70-120), the caller copies
// those it wants out of `regs`.
#if defined(__CUDACC__)
__host__ __device__
#endif
inline void vm_run(const u32 *code, const u32 *fn_info, u32 fn, u32 *regs, const u32 *consts32, u32 *result, const FrParams &P,
                   int &err, u32 &ret_base, u32 &ret_cnt) {
    FnInfo fi = vm_fn(fn_info, fn);
    const u32 *ins = code + 5 * (size_t)fi.code_off;
    u32 *fr = regs;          // registers of the running frame
    u32 base = 0, depth = 0;
    VmFrame stack[VM_MAX_DEPTH];
    u32 pc = 0;
    u256_set_u32(result, 0);
    ret_base = 0;
    ret_cnt = 0;
    for (u32 step = 0; step < (u32)VM_MAX_STEPS; ++step) {
        if (pc >= fi.n_instr) { err = 2; return; }
        const u32 op = ins[5 * pc], d = ins[5 * pc + 1], a = ins[5 * pc + 2], b = ins[5 * pc + 3], c = ins[5 * pc + 4];
        ++pc;
        u32 va[8], vb[8], vc[8], r[8];
        if (op == FOP_JMP) { pc = a & 0x3FFFFFFFu; continue; }
        if (op == OP_CALL) {   // a nested call: new frame behind this one, arguments copied, the rest zero
            const u32 f = a & 0x3FFFFFFFu;
            const FnInfo callee = vm_fn(fn_info, f);
            const u32 nb = base + fi.n_regs;
            if (depth >= (u32)VM_MAX_DEPTH || nb + callee.n_regs > (u32)VM_MAX_REGS) { err = 2; return; }
            u32 *nf = regs + 8 * (size_t)nb;
            for (u32 k = 0; k < callee.n_params * 8; ++k) nf[k] = fr[8 * (size_t)b + k];
            for (u32 k = callee.n_params * 8; k < callee.n_regs * 8; ++k) nf[k] = 0;
            stack[depth].fn = fn; stack[depth].pc = pc; stack[depth].base = base; stack[depth].dst = d;
            stack[depth].want = c & 0x3FFFFFFFu;
            ++depth;
            fn = f; fi = callee; ins = code + 5 * (size_t)fi.code_off; base = nb; fr = nf; pc = 0;
            continue;
        }
        vm_operand(va, a, fr, consts32);
        if (op == FOP_JZ) { if (u256_is_zero(va)) pc = b & 0x3FFFFFFFu; continue; }
        if (op == FOP_RET) {
            const u32 cnt = b & 0x3FFFFFFFu;
            if (depth == 0) {
                u256_set(result, va);
                ret_cnt = cnt;
                if (ret_cnt > 1) ret_base = a;   // (the lowering checked: a register, a + count <= n_regs)
                return;
            }
            --depth;
            const VmFrame &top = stack[depth];
            u32 *cf = regs + 8 * (size_t)top.base;   // the caller's registers
            const u32 want = top.want > 1 ? top.want : 1u;
            if (want > 1 && cnt < want) { err = 2; return; }
            if (cnt > 1) {
                for (u32 k = 0; k < want * 8; ++k) cf[8 * (size_t)top.dst + k] = fr[8 * (size_t)a + k];
            } else {
                for (int k = 0; k < 8; ++k) cf[8 * (size_t)top.dst + k] = va[k];
            }
            fn = top.fn; fi = vm_fn(fn_info, fn); ins = code + 5 * (size_t)fi.code_off; base = top.base; fr = cf; pc = top.pc;
            continue;
        }
        vm_operand(vb, b, fr, consts32);
        if (op == FOP_LOADX) {
            int i = vm_index(vb, a & 0x3FFFFFFFu, c & 0x3FFFFFFFu);
            if (i < 0) { err = 2; return; }
            for (int k = 0; k < 8; ++k) fr[8 * (size_t)d + k] = fr[8 * (size_t)i + k];
            continue;
        }
        vm_operand(vc, c, fr, consts32);
        if (op == FOP_STOREX) {
            int i = vm_index(vb, a & 0x3FFFFFFFu, d & 0x3FFFFFFFu);
            if (i < 0) { err = 2; return; }
            for (int k = 0; k < 8; ++k) fr[8 * (size_t)i + k] = vc[k];
            continue;
        }
        int e = 0;
        fr_apply_canonical(op, r, va, vb, vc, P, e);
        if (e) err = 1;
        for (int k = 0; k < 8; ++k) fr[8 * (size_t)d + k] = r[k];
    }
    err = 2;
}

// ---- the narrow register machine -------------------------------------------------------------------------------
// Hint functions are limb arithmetic: their values are 64-bit limbs, carries, products of two limbs, loop counters.  A
// call frame of 32-byte registers in local memory is what a call costs (hundreds of concurrent calls per SM), so a
// call first runs on a machine whose registers are 128-bit integers (16 bytes, half the frame and half the traffic per
// instruction; plain integer add / multiply / compare instead of modular ones).  A value below 2^128 is its own
// canonical form and is non-negative in the signed view of every supported prime (all above 2^250), so the integer
// result IS the field result as long as it stays below 2^128.  Anything else - a wider argument or constant, a sum or
// product that leaves 128 bits, a difference below zero, an operator the narrow machine does not have (field division,
// powers, bit complement) - abandons the run: the caller repeats the call on the full-width machine (functions are pure,
// nothing was stored).  Errors (bad index, runaway loop) are reported as on the full-width machine.
struct N128 {
    u64 lo, hi;
};
CW_HD void mul64wide_vm(u64 a, u64 b, u64 &lo, u64 &hi) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umul64hi(a, b);
#else
    unsigned __int128 p = (unsigned __int128)a * b;
    lo = (u64)p;
    hi = (u64)(p >> 64);
#endif
}
CW_HD bool vmn_operand(N128 &v, u32 o, const u32 *regs, const u32 *consts32) {
    if (o & 0x80000000u) {
        const u32 *p = consts32 + 8 * (size_t)(o & 0x3FFFFFFFu);
        if (p[4] | p[5] | p[6] | p[7]) return false;
        v.lo = p[0] | ((u64)p[1] << 32);
        v.hi = p[2] | ((u64)p[3] << 32);
    } else if (o & 0x40000000u) {
        v.lo = o & 0x3FFFFFFFu;
        v.hi = 0;
    } else {
        const u32 *p = regs + 4 * (size_t)o;
        v.lo = p[0] | ((u64)p[1] << 32);
        v.hi = p[2] | ((u64)p[3] << 32);
    }
    return true;
}
CW_HD void vmn_store(u32 *regs, u32 d, const N128 &v) {
    u32 *p = regs + 4 * (size_t)d;
    p[0] = (u32)v.lo; p[1] = (u32)(v.lo >> 32); p[2] = (u32)v.hi; p[3] = (u32)(v.hi >> 32);
}
CW_HD bool n128_lt(const N128 &a, const N128 &b) { return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo); }
CW_HD bool n128_eq(const N128 &a, const N128 &b) { return a.hi == b.hi && a.lo == b.lo; }
// one value operator on 128-bit integers; false: the result (or the operator) needs the full-width machine
CW_HD bool vmn_apply(u32 op, N128 &r, const N128 &a, const N128 &b, const N128 &c) {
    switch (op) {
        case OP_ADD: {
            r.lo = a.lo + b.lo;
            const u64 cy = r.lo < a.lo ? 1u : 0u;
            const u64 t = a.hi + b.hi;
            r.hi = t + cy;
            return !(t < a.hi || r.hi < t);
        }
        case OP_SUB: {
            if (n128_lt(a, b)) return false;   // negative: q - (b - a)
            r.lo = a.lo - b.lo;
            r.hi = a.hi - b.hi - (a.lo < b.lo ? 1u : 0u);
            return true;
        }
        case OP_MUL: {
            if (a.hi && b.hi) return false;
            const N128 &x = a.hi ? a : b, &y = a.hi ? b : a;   // y.hi == 0
            u64 lo, hi, clo, chi;
            mul64wide_vm(x.lo, y.lo, lo, hi);
            mul64wide_vm(x.hi, y.lo, clo, chi);
            if (chi) return false;
            r.lo = lo;
            r.hi = hi + clo;
            return r.hi >= hi;
        }
        case OP_IDIV: case OP_MOD:
            if (a.hi | b.hi || !b.lo) return false;   // (division by zero: reported by the full-width machine)
            r.lo = op == OP_IDIV ? a.lo / b.lo : a.lo % b.lo;
            r.hi = 0;
            return true;
        case OP_SHR: {
            if (b.hi || b.lo >= 128u) return false;
            const u32 k = (u32)b.lo;
            if (k == 0) r = a;
            else if (k < 64u) { r.lo = (a.lo >> k) | (a.hi << (64u - k)); r.hi = a.hi >> k; }
            else { r.lo = a.hi >> (k - 64u); r.hi = 0; }
            return true;
        }
        case OP_SHL: {
            if (b.hi || b.lo >= 128u) return false;
            const u32 k = (u32)b.lo;
            if (k == 0) { r = a; return true; }
            if (k < 64u) {
                if (a.hi >> (64u - k)) return false;
                r.hi = (a.hi << k) | (a.lo >> (64u - k));
                r.lo = a.lo << k;
            } else {
                if (a.hi || (k > 64u && (a.lo >> (128u - k)))) return false;
                r.hi = a.lo << (k - 64u);
                r.lo = 0;
            }
            return true;
        }
        case OP_LEQ: r.lo = !n128_lt(b, a); r.hi = 0; return true;
        case OP_GEQ: r.lo = !n128_lt(a, b); r.hi = 0; return true;
        case OP_LT: r.lo = n128_lt(a, b); r.hi = 0; return true;
        case OP_GT: r.lo = n128_lt(b, a); r.hi = 0; return true;
        case OP_EQ: r.lo = n128_eq(a, b); r.hi = 0; return true;
        case OP_NEQ: r.lo = !n128_eq(a, b); r.hi = 0; return true;
        case OP_LOR: r.lo = ((a.lo | a.hi) || (b.lo | b.hi)) ? 1u : 0u; r.hi = 0; return true;
        case OP_LAND: r.lo = ((a.lo | a.hi) && (b.lo | b.hi)) ? 1u : 0u; r.hi = 0; return true;
        case OP_LNOT: r.lo = (a.lo | a.hi) ? 0u : 1u; r.hi = 0; return true;
        case OP_BOR: r.lo = a.lo | b.lo; r.hi = a.hi | b.hi; return true;
        case OP_BAND: r.lo = a.lo & b.lo; r.hi = a.hi & b.hi; return true;
        case OP_BXOR: r.lo = a.lo ^ b.lo; r.hi = a.hi ^ b.hi; return true;
        case OP_NEG: if (a.lo | a.hi) return false; r = a; return true;
        case OP_COPY: r = a; return true;
        case OP_SELECT: r = (c.lo | c.hi) ? a : b; return true;
        default: return false;
    }
}
// regs: the arguments in the full-width layout (8 words per register, as the caller loads them); they are repacked to 4
// words in place.  Returns false when the call has to be repeated on the full-width machine (regs are garbage then).
// On success: err / result / ret_base / ret_cnt as vm_run; returned registers are 4 words each (vmn_result).
#if defined(__CUDACC__)
__host__ __device__
#endif
inline bool vm_run_narrow(const u32 *code, const u32 *fn_info, u32 fn, u32 *regs, const u32 *consts32, u32 *result, int &err,
                          u32 &ret_base, u32 &ret_cnt) {
    FnInfo fi = vm_fn(fn_info, fn);
    for (u32 k = 0; k < fi.n_params; ++k) {
        const u32 *p = regs + 8 * (size_t)k;
        if (p[4] | p[5] | p[6] | p[7]) return false;
    }
    for (u32 k = 0; k < fi.n_params; ++k)
        for (int j = 0; j < 4; ++j) regs[4 * (size_t)k + j] = regs[8 * (size_t)k + j];
    for (u32 k = 4 * fi.n_params; k < 4 * fi.n_regs; ++k) regs[k] = 0;
    const u32 *ins = code + 5 * (size_t)fi.code_off;
    u32 *fr = regs;
    u32 base = 0, depth = 0;
    VmFrame stack[VM_MAX_DEPTH];
    u32 pc = 0;
    u256_set_u32(result, 0);
    ret_base = 0;
    ret_cnt = 0;
    for (u32 step = 0; step < (u32)VM_MAX_STEPS; ++step) {
        if (pc >= fi.n_instr) { err = 2; return true; }
        const u32 op = ins[5 * pc], d = ins[5 * pc + 1], a = ins[5 * pc + 2], b = ins[5 * pc + 3], c = ins[5 * pc + 4];
        ++pc;
        if (op == FOP_JMP) { pc = a & 0x3FFFFFFFu; continue; }
        if (op == OP_CALL) {
            const u32 f = a & 0x3FFFFFFFu;
            const FnInfo callee = vm_fn(fn_info, f);
            const u32 nb = base + fi.n_regs;
            if (depth >= (u32)VM_MAX_DEPTH || nb + callee.n_regs > (u32)VM_MAX_REGS) { err = 2; return true; }
            u32 *nf = regs + 4 * (size_t)nb;
            for (u32 k = 0; k < callee.n_params * 4; ++k) nf[k] = fr[4 * (size_t)b + k];
            for (u32 k = callee.n_params * 4; k < callee.n_regs * 4; ++k) nf[k] = 0;
            stack[depth].fn = fn; stack[depth].pc = pc; stack[depth].base = base; stack[depth].dst = d;
            stack[depth].want = c & 0x3FFFFFFFu;
            ++depth;
            fn = f; fi = callee; ins = code + 5 * (size_t)fi.code_off; base = nb; fr = nf; pc = 0;
            continue;
        }
        N128 va, vb, vc, r;
        if (!vmn_operand(va, a, fr, consts32)) return false;
        if (op == FOP_JZ) { if (!(va.lo | va.hi)) pc = b & 0x3FFFFFFFu; continue; }
        if (op == FOP_RET) {
            const u32 cnt = b & 0x3FFFFFFFu;
            if (depth == 0) {
                result[0] = (u32)va.lo; result[1] = (u32)(va.lo >> 32); result[2] = (u32)va.hi; result[3] = (u32)(va.hi >> 32);
                ret_cnt = cnt;
                if (ret_cnt > 1) ret_base = a;
                return true;
            }
            --depth;
            const VmFrame &top = stack[depth];
            u32 *cf = regs + 4 * (size_t)top.base;
            const u32 want = top.want > 1 ? top.want : 1u;
            if (want > 1 && cnt < want) { err = 2; return true; }
            if (cnt > 1) {
                for (u32 k = 0; k < want * 4; ++k) cf[4 * (size_t)top.dst + k] = fr[4 * (size_t)a + k];
            } else vmn_store(cf, top.dst, va);
            fn = top.fn; fi = vm_fn(fn_info, fn); ins = code + 5 * (size_t)fi.code_off; base = top.base; fr = cf; pc = top.pc;
            continue;
        }
        if (!vmn_operand(vb, b, fr, consts32)) return false;
        if (op == FOP_LOADX || op == FOP_STOREX) {
            const u32 ab = a & 0x3FFFFFFFu, limit = (op == FOP_LOADX ? c : d) & 0x3FFFFFFFu;
            if (vb.hi || (vb.lo >> 32) || vb.lo + ab >= limit) { err = 2; return true; }
            const u32 i = (u32)vb.lo + ab;
            if (op == FOP_LOADX) {
                for (int k = 0; k < 4; ++k) fr[4 * (size_t)d + k] = fr[4 * (size_t)i + k];
            } else {
                if (!vmn_operand(vc, c, fr, consts32)) return false;
                vmn_store(fr, i, vc);
            }
            continue;
        }
        if (!vmn_operand(vc, c, fr, consts32)) return false;
        if (!vmn_apply(op, r, va, vb, vc)) return false;
        vmn_store(fr, d, r);
    }
    err = 2;
    return true;
}
// register `reg` of a finished call as a canonical element (narrow: 4 stored words, the upper half is zero)
CW_HD void vm_result(u32 *out, const u32 *regs, u32 reg, bool narrow) {
    if (narrow) {
        for (int k = 0; k < 4; ++k) { out[k] = regs[4 * (size_t)reg + k]; out[4 + k] = 0; }
    } else {
        for (int k = 0; k < 8; ++k) out[k] = regs[8 * (size_t)reg + k];
    }
}

}  // namespace cw
