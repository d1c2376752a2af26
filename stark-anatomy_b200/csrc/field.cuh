// field.cuh -- arithmetic in F_p, p = 1 + 407 * 2^119 (reference: code/algebra.py:65-98).
//
// One element = 16 bytes = four little-endian 32-bit limbs of the canonical
// residue in [0, p).  Everything here is __host__ __device__ so that the exact
// code the kernels run can be exercised on the CPU by tests/emu (thread-by-thread
// emulation of the kernels' phase functions).
//
// Multiplication is Montgomery (R = 2^128) specialised to this prime:
//   p = 1 + P3 * 2^96 with P3 = 407 << 23 = 0xCB800000, so p^-1 mod 2^128 = 1 - P3 * 2^96.
//   The device code reduces with +p^-1: m = t_lo * p^-1 mod 2^128 is t_lo with (t0 * P3 mod 2^32) taken
//   off its top word, and t * 2^-128 = t_hi - ((m * P3) >> 32) - borrow, in (-p, p): four multiplies by
//   the constant P3 and one masked add of p (fe_montmul below).  The portable version (host, tests/emu,
//   sa_selftest_field) uses the textbook -p^-1 form, m = ((t0 * P3 mod 2^32) << 96) - t_lo; both return the
//   canonical residue of a * b * 2^-128.
// Twiddles are stored pre-multiplied by R ("Montgomery form"), data stays in
// canonical form: montmul(x, w*R) = x*w, so no conversion passes are needed and
// every result is the canonical residue the reference's Python ints produce.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SA_HD __host__ __device__ __forceinline__
#define SA_HDC __host__ __device__ static constexpr
#define SA_ALIGN16 __align__(16)
#else
#define SA_HD inline
#define SA_HDC static constexpr
#define SA_ALIGN16 alignas(16)
#endif

namespace sa {

struct SA_ALIGN16 fe {
    uint32_t v[4];
};

static constexpr uint32_t P3 = 0xCB800000u;  // top limb of p; low limbs are (1, 0, 0)

SA_HD fe fe_make(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3) {
    fe r;
    r.v[0] = a0; r.v[1] = a1; r.v[2] = a2; r.v[3] = a3;
    return r;
}
SA_HD fe fe_zero() { return fe_make(0, 0, 0, 0); }
SA_HD fe fe_one() { return fe_make(1, 0, 0, 0); }
SA_HD fe fe_mont_one() { return fe_make(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0x347FFFFFu); }  // R mod p, R = 2^128
SA_HD fe fe_r2() { return fe_make(0x0E778236u, 0x5BD53A7Fu, 0x1A6AEDC2u, 0xAAF4AD9Au); }  // R^2 mod p
SA_HD fe fe_from_u64(uint64_t x) { return fe_make((uint32_t)x, (uint32_t)(x >> 32), 0, 0); }
SA_HD bool fe_is_zero(const fe &a) { return (a.v[0] | a.v[1] | a.v[2] | a.v[3]) == 0; }
SA_HD bool fe_eq(const fe &a, const fe &b) {
    return ((a.v[0] ^ b.v[0]) | (a.v[1] ^ b.v[1]) | (a.v[2] ^ b.v[2]) | (a.v[3] ^ b.v[3])) == 0;
}

// r = (s + carry * 2^128) reduced once: subtract p when the 129-bit value is >= p.
SA_HD fe fe_cond_sub_p_portable(uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t carry) {
    uint64_t t = (uint64_t)s0 - 1u;
    uint32_t d0 = (uint32_t)t;
    uint32_t br = (uint32_t)(t >> 63);
    t = (uint64_t)s1 - br;
    uint32_t d1 = (uint32_t)t;
    br = (uint32_t)(t >> 63);
    t = (uint64_t)s2 - br;
    uint32_t d2 = (uint32_t)t;
    br = (uint32_t)(t >> 63);
    t = (uint64_t)s3 - P3 - br;
    uint32_t d3 = (uint32_t)t;
    br = (uint32_t)(t >> 63);
    bool use = (carry != 0) | (br == 0);
    return fe_make(use ? d0 : s0, use ? d1 : s1, use ? d2 : s2, use ? d3 : s3);
}

// algebra.py:78-79
SA_HD fe fe_add_portable(const fe &a, const fe &b) {
    uint64_t c = (uint64_t)a.v[0] + b.v[0];
    uint32_t s0 = (uint32_t)c;
    c = (c >> 32) + a.v[1] + b.v[1];
    uint32_t s1 = (uint32_t)c;
    c = (c >> 32) + a.v[2] + b.v[2];
    uint32_t s2 = (uint32_t)c;
    c = (c >> 32) + a.v[3] + b.v[3];
    uint32_t s3 = (uint32_t)c;
    return fe_cond_sub_p_portable(s0, s1, s2, s3, (uint32_t)(c >> 32));
}

// algebra.py:81-82
SA_HD fe fe_sub_portable(const fe &a, const fe &b) {
    uint64_t t = (uint64_t)a.v[0] - b.v[0];
    uint32_t d0 = (uint32_t)t;
    uint32_t br = (uint32_t)(t >> 63);
    t = (uint64_t)a.v[1] - b.v[1] - br;
    uint32_t d1 = (uint32_t)t;
    br = (uint32_t)(t >> 63);
    t = (uint64_t)a.v[2] - b.v[2] - br;
    uint32_t d2 = (uint32_t)t;
    br = (uint32_t)(t >> 63);
    t = (uint64_t)a.v[3] - b.v[3] - br;
    uint32_t d3 = (uint32_t)t;
    br = (uint32_t)(t >> 63);
    // borrow -> add p = (1, 0, 0, P3)
    uint64_t c = (uint64_t)d0 + br;
    uint32_t r0 = (uint32_t)c;
    c = (c >> 32) + d1;
    uint32_t r1 = (uint32_t)c;
    c = (c >> 32) + d2;
    uint32_t r2 = (uint32_t)c;
    uint32_t r3 = (uint32_t)(c >> 32) + d3 + (br ? P3 : 0u);
    return fe_make(r0, r1, r2, r3);
}

// Montgomery product a * b * 2^-128 mod p, canonical output, inputs < p.
SA_HD fe fe_montmul_portable(const fe &a, const fe &b) {
    uint32_t t[8];
    uint64_t c;
    // 4x4 schoolbook, operand scanning; every accumulation fits 64 bits
    c = (uint64_t)a.v[0] * b.v[0];
    t[0] = (uint32_t)c;
    c = (c >> 32) + (uint64_t)a.v[0] * b.v[1];
    t[1] = (uint32_t)c;
    c = (c >> 32) + (uint64_t)a.v[0] * b.v[2];
    t[2] = (uint32_t)c;
    c = (c >> 32) + (uint64_t)a.v[0] * b.v[3];
    t[3] = (uint32_t)c;
    t[4] = (uint32_t)(c >> 32);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 1; i < 4; i++) {
        c = (uint64_t)a.v[i] * b.v[0] + t[i];
        t[i] = (uint32_t)c;
        c = (c >> 32) + (uint64_t)a.v[i] * b.v[1] + t[i + 1];
        t[i + 1] = (uint32_t)c;
        c = (c >> 32) + (uint64_t)a.v[i] * b.v[2] + t[i + 2];
        t[i + 2] = (uint32_t)c;
        c = (c >> 32) + (uint64_t)a.v[i] * b.v[3] + t[i + 3];
        t[i + 3] = (uint32_t)c;
        t[i + 4] = (uint32_t)(c >> 32);
    }
    // m = ((t0*P3 mod 2^32) << 96) - t_lo  (mod 2^128);  u = m * P3 (160 bits)
    uint32_t m0 = 0u - t[0];
    uint64_t u = (uint64_t)m0 * P3;
    uint32_t u0 = (uint32_t)u;
    uint32_t x = 0u - u0;  // = t0 * P3 mod 2^32
    uint32_t bw = (t[0] != 0u);
    uint64_t s = (uint64_t)0 - t[1] - bw;
    uint32_t m1 = (uint32_t)s;
    bw = (uint32_t)(s >> 63);
    s = (uint64_t)0 - t[2] - bw;
    uint32_t m2 = (uint32_t)s;
    bw = (uint32_t)(s >> 63);
    s = (uint64_t)x - t[3] - bw;
    uint32_t m3 = (uint32_t)s;
    uint32_t ca = (uint32_t)(s >> 63);  // carry of t_lo + m
    uint32_t cb = (u0 != 0u);           // carry of (x + u0) << 96
    u = (u >> 32) + (uint64_t)m1 * P3;
    uint32_t u1 = (uint32_t)u;
    u = (u >> 32) + (uint64_t)m2 * P3;
    uint32_t u2 = (uint32_t)u;
    u = (u >> 32) + (uint64_t)m3 * P3;
    uint32_t u3 = (uint32_t)u;
    uint32_t u4 = (uint32_t)(u >> 32);
    // r = t_hi + (u1..u4) + ca + cb  < 2p
    c = (uint64_t)t[4] + u1 + ca + cb;
    uint32_t r0 = (uint32_t)c;
    c = (c >> 32) + t[5] + u2;
    uint32_t r1 = (uint32_t)c;
    c = (c >> 32) + t[6] + u3;
    uint32_t r2 = (uint32_t)c;
    c = (c >> 32) + t[7] + u4;
    uint32_t r3 = (uint32_t)c;
    return fe_cond_sub_p_portable(r0, r1, r2, r3, (uint32_t)(c >> 32));
}

#if defined(__CUDA_ARCH__) && !defined(SA_PORTABLE_FIELD)
// ---- sm_100a versions: explicit carry chains.  ptxas fuses each
// mad.lo.cc/madc.hi.cc pair into one IMAD.WIDE.U32(.X) with a predicate carry,
// so the 4x4 product is 16 wide multiply-adds and the reduction 5 more.
// SASS per operation (tools/sass_mix.py): montmul 21 IMAD.WIDE + ~13 IMAD + ~24 ALU, add 13 ALU,
// sub 7 ALU + 3 IMAD.
__device__ __forceinline__ fe fe_cond_sub_p(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3, uint32_t top) {
    uint32_t d0, d1, d2, d3, br;
    asm("sub.cc.u32 %0, %5, 1;\n\t"
        "subc.cc.u32 %1, %6, 0;\n\t"
        "subc.cc.u32 %2, %7, 0;\n\t"
        "subc.cc.u32 %3, %8, 0xCB800000;\n\t"
        "subc.u32 %4, 0, 0;"
        : "=r"(d0), "=r"(d1), "=r"(d2), "=r"(d3), "=r"(br)
        : "r"(r0), "r"(r1), "r"(r2), "r"(r3));
    bool use = (top != 0) | (br == 0);
    return fe_make(use ? d0 : r0, use ? d1 : r1, use ? d2 : r2, use ? d3 : r3);
}
// (d3..d0) + p when m is all-ones, unchanged when m is zero (m = the borrow word of a subtraction that
// went negative).  The two mask words (1 and P3, or zeros) are products of the all-ones word, so they
// issue on the FMA pipe rather than the ALU pipe.  Measured on the 16 x 2^20 NTT step
// (profiles/r01g_field_v2.txt): montmul's w an AND and both add-backs multiplies (the form used here)
// 0.737 ms; all three multiplies 0.741; only fe_sub's add-back an AND 0.748; all three ANDs 0.758.
__device__ __forceinline__ fe fe_cond_add_p(uint32_t d0, uint32_t d1, uint32_t d2, uint32_t d3, uint32_t m) {
    uint32_t p0, p3;
    asm("mul.lo.u32 %0, %2, %2;\n\t"           // (-1)^2 = 1
        "mul.lo.u32 %1, %2, 0x34800000;"        // (-1) * (-P3) = P3
        : "=r"(p0), "=r"(p3) : "r"(m));
    uint32_t r0, r1, r2, r3;
    asm("add.cc.u32 %0, %4, %8;\n\t"
        "addc.cc.u32 %1, %5, 0;\n\t"
        "addc.cc.u32 %2, %6, 0;\n\t"
        "addc.u32 %3, %7, %9;"
        : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
        : "r"(d0), "r"(d1), "r"(d2), "r"(d3), "r"(p0), "r"(p3));
    return fe_make(r0, r1, r2, r3);
}
// a five-limb sum, the trial subtraction of p and a predicated select: 13 ALU instructions (the
// a - (p - b) form with the masked add-back needs 14 plus two multiplies, and ptxas does not fuse
// a + b + (2^128 - p) into three-input IADD3 chains)
__device__ __forceinline__ fe fe_add(const fe &a, const fe &b) {
    uint32_t s0, s1, s2, s3, c;
    asm("add.cc.u32 %0, %5, %9;\n\t"
        "addc.cc.u32 %1, %6, %10;\n\t"
        "addc.cc.u32 %2, %7, %11;\n\t"
        "addc.cc.u32 %3, %8, %12;\n\t"
        "addc.u32 %4, 0, 0;"
        : "=r"(s0), "=r"(s1), "=r"(s2), "=r"(s3), "=r"(c)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]),
          "r"(b.v[3]));
    return fe_cond_sub_p(s0, s1, s2, s3, c);
}
__device__ __forceinline__ fe fe_sub(const fe &a, const fe &b) {
    uint32_t d0, d1, d2, d3, m;
    asm("sub.cc.u32 %0, %5, %9;\n\t"
        "subc.cc.u32 %1, %6, %10;\n\t"
        "subc.cc.u32 %2, %7, %11;\n\t"
        "subc.cc.u32 %3, %8, %12;\n\t"
        "subc.u32 %4, 0, 0;"
        : "=r"(d0), "=r"(d1), "=r"(d2), "=r"(d3), "=r"(m)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]),
          "r"(b.v[3]));
    return fe_cond_add_p(d0, d1, d2, d3, m);
}
__device__ __forceinline__ fe fe_montmul(const fe &a, const fe &b) {
    uint32_t a0 = a.v[0], a1 = a.v[1], a2 = a.v[2], a3 = a.v[3];
    uint32_t b0 = b.v[0], b1 = b.v[1], b2 = b.v[2], b3 = b.v[3];
    // e = sum of a_i*b_j with i+j even (word aligned), o = the i+j odd ones one word down
    uint32_t e0, e1, e2, e3, e4, e5, e6, e7, o0, o1, o2, o3, o4, o5, o6;
    asm("{\n\t"
        "mul.lo.u32 %0, %15, %19;\n\t"  // e0:e1 = a0*b0
        "mul.hi.u32 %1, %15, %19;\n\t"
        "mul.lo.u32 %2, %15, %21;\n\t"  // e2:e3 = a0*b2
        "mul.hi.u32 %3, %15, %21;\n\t"
        "mul.lo.u32 %8, %15, %20;\n\t"  // o0:o1 = a0*b1
        "mul.hi.u32 %9, %15, %20;\n\t"
        "mul.lo.u32 %10, %15, %22;\n\t"  // o2:o3 = a0*b3
        "mul.hi.u32 %11, %15, %22;\n\t"
        "mad.lo.cc.u32 %2, %16, %20, %2;\n\t"  // a1: (1,1)@2 (1,3)@4
        "madc.hi.cc.u32 %3, %16, %20, %3;\n\t"
        "madc.lo.cc.u32 %4, %16, %22, 0;\n\t"
        "madc.hi.u32 %5, %16, %22, 0;\n\t"
        "mad.lo.cc.u32 %8, %16, %19, %8;\n\t"  // a1: (1,0)@1 (1,2)@3
        "madc.hi.cc.u32 %9, %16, %19, %9;\n\t"
        "madc.lo.cc.u32 %10, %16, %21, %10;\n\t"
        "madc.hi.cc.u32 %11, %16, %21, %11;\n\t"
        "addc.u32 %12, 0, 0;\n\t"
        "mad.lo.cc.u32 %2, %17, %19, %2;\n\t"  // a2: (2,0)@2 (2,2)@4
        "madc.hi.cc.u32 %3, %17, %19, %3;\n\t"
        "madc.lo.cc.u32 %4, %17, %21, %4;\n\t"
        "madc.hi.cc.u32 %5, %17, %21, %5;\n\t"
        "addc.u32 %6, 0, 0;\n\t"
        "mad.lo.cc.u32 %10, %17, %20, %10;\n\t"  // a2: (2,1)@3 (2,3)@5
        "madc.hi.cc.u32 %11, %17, %20, %11;\n\t"
        "madc.lo.cc.u32 %12, %17, %22, %12;\n\t"
        "madc.hi.u32 %13, %17, %22, 0;\n\t"
        "mad.lo.cc.u32 %4, %18, %20, %4;\n\t"  // a3: (3,1)@4 (3,3)@6
        "madc.hi.cc.u32 %5, %18, %20, %5;\n\t"
        "madc.lo.cc.u32 %6, %18, %22, %6;\n\t"
        "madc.hi.u32 %7, %18, %22, 0;\n\t"
        "mad.lo.cc.u32 %10, %18, %19, %10;\n\t"  // a3: (3,0)@3 (3,2)@5
        "madc.hi.cc.u32 %11, %18, %19, %11;\n\t"
        "madc.lo.cc.u32 %12, %18, %21, %12;\n\t"
        "madc.hi.cc.u32 %13, %18, %21, %13;\n\t"
        "addc.u32 %14, 0, 0;\n\t"
        "add.cc.u32 %1, %1, %8;\n\t"  // t = e + (o << 32)
        "addc.cc.u32 %2, %2, %9;\n\t"
        "addc.cc.u32 %3, %3, %10;\n\t"
        "addc.cc.u32 %4, %4, %11;\n\t"
        "addc.cc.u32 %5, %5, %12;\n\t"
        "addc.cc.u32 %6, %6, %13;\n\t"
        "addc.u32 %7, %7, %14;\n\t"
        "}"
        : "=&r"(e0), "=&r"(e1), "=&r"(e2), "=&r"(e3), "=&r"(e4), "=&r"(e5), "=&r"(e6), "=&r"(e7),
          "=&r"(o0), "=&r"(o1), "=&r"(o2), "=&r"(o3), "=&r"(o4), "=&r"(o5), "=&r"(o6)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(b2), "r"(b3));
    (void)o0; (void)o1; (void)o2; (void)o3; (void)o4; (void)o5; (void)o6;
    // Reduction with p^-1 = 1 - P3*2^96 (mod 2^128) instead of -p^-1: m = t_lo * p^-1 mod 2^128 is t_lo
    // with (t0*P3 mod 2^32) taken off its top word, and since t_lo - m and m*P3*2^96 cancel below bit
    // 128,  t*2^-128 = t_hi - ((m*P3) >> 32) - w  (w = the borrow of that top word), in (-p, p): one
    // masked add of p.  Half the ALU instructions of the m = -t_lo form (no 128-bit negation, no
    // five-way select); the add-back's mask words come from multiplies so that they issue on the FMA
    // pipe, while w is an AND (the fastest split, see fe_cond_add_p).
    uint32_t x = e0 * P3;
    uint32_t m3, nw;
    asm("sub.cc.u32 %0, %2, %3;\n\t"
        "subc.u32 %1, 0, 0;"
        : "=r"(m3), "=r"(nw)
        : "r"(e3), "r"(x));
    const uint32_t w = nw & 1u;
    uint32_t u1, u2, u3, u4;
    asm("mad.hi.u32 %0, %4, 0xCB800000, %8;\n\t"
        "mad.lo.cc.u32 %0, %5, 0xCB800000, %0;\n\t"
        "madc.hi.u32 %1, %5, 0xCB800000, 0;\n\t"
        "mad.lo.cc.u32 %1, %6, 0xCB800000, %1;\n\t"
        "madc.hi.u32 %2, %6, 0xCB800000, 0;\n\t"
        "mad.lo.cc.u32 %2, %7, 0xCB800000, %2;\n\t"
        "madc.hi.u32 %3, %7, 0xCB800000, 0;"
        : "=&r"(u1), "=&r"(u2), "=&r"(u3), "=&r"(u4)
        : "r"(e0), "r"(e1), "r"(e2), "r"(m3), "r"(w));
    uint32_t r0, r1, r2, r3, top;
    asm("sub.cc.u32 %0, %5, %9;\n\t"
        "subc.cc.u32 %1, %6, %10;\n\t"
        "subc.cc.u32 %2, %7, %11;\n\t"
        "subc.cc.u32 %3, %8, %12;\n\t"
        "subc.u32 %4, 0, 0;"
        : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(top)
        : "r"(e4), "r"(e5), "r"(e6), "r"(e7), "r"(u1), "r"(u2), "r"(u3), "r"(u4));
    return fe_cond_add_p(r0, r1, r2, r3, top);
}
#else
SA_HD fe fe_add(const fe &a, const fe &b) { return fe_add_portable(a, b); }
SA_HD fe fe_sub(const fe &a, const fe &b) { return fe_sub_portable(a, b); }
SA_HD fe fe_montmul(const fe &a, const fe &b) { return fe_montmul_portable(a, b); }
#endif
// algebra.py:84-85
SA_HD fe fe_neg(const fe &a) { return fe_sub(fe_zero(), a); }

SA_HD fe fe_to_mont(const fe &a) { return fe_montmul(a, fe_r2()); }
SA_HD fe fe_from_mont(const fe &a) { return fe_montmul(a, fe_one()); }
// algebra.py:75-76 (canonical in, canonical out)
SA_HD fe fe_mul(const fe &a, const fe &b) { return fe_montmul(fe_to_mont(a), b); }

// base in Montgomery form, result in Montgomery form; e < 2^64
SA_HD fe fe_mont_pow_u64(const fe &base_m, uint64_t e) {
    fe acc = fe_mont_one();
    fe b = base_m;
    while (e) {
        if (e & 1) acc = fe_montmul(acc, b);
        b = fe_montmul(b, b);
        e >>= 1;
    }
    return acc;
}

// a^(p-2) with a in Montgomery form, result in Montgomery form (0 -> 0, as
// algebra.py:87-89's xgcd route gives for a zero operand).
// p - 2 = 0xCB7FFFFF FFFFFFFF FFFFFFFF FFFFFFFF
SA_HD fe fe_mont_inv(const fe &a_m) {
    // left-to-right over the 128 exponent bits
    const uint32_t e[4] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xCB7FFFFFu};
    fe acc = fe_mont_one();
    for (int w = 3; w >= 0; w--) {
        for (int bit = 31; bit >= 0; bit--) {
            acc = fe_montmul(acc, acc);
            if ((e[w] >> bit) & 1u) acc = fe_montmul(acc, a_m);
        }
    }
    return acc;
}

}  // namespace sa
