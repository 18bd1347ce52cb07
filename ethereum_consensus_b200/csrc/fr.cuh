// Fr: the BLS12-381 scalar field (r = 0x73eda753...00000001, 255 bits), 8 x 32-bit limbs, Montgomery form with
// R = 2^256.  The field of KZG blob elements, evaluation points and the scalars of the G1 combinations (kzg.cu).
//
// Like fp.cuh the same source compiles for the host (tests/host_math/host_kzg.cpp checks it against Python ints).
// r leaves a single spare bit (2r < 2^256), so every result is kept fully reduced: the lazy [0, 2p) scheme of fpl.cuh
// needs headroom this field does not have.
#pragma once
#include <cstdint>

#include "fp.cuh"   // B200_HD

namespace b200 {

struct Fr {
    uint32_t l[8];
};

#define B200_FR_R {{0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u, 0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u}}
#define B200_FR_ONE {{0xfffffffeu, 0x00000001u, 0x00034802u, 0x5884b7fau, 0xecbc4ff5u, 0x998c4fefu, 0xacc5056fu, 0x1824b159u}}
#define B200_FR_R2 {{0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu, 0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u}}
// -r^-1 mod 2^32 (r = 1 mod 2^32)
#define B200_FR_N0 0xffffffffu
// the primitive 4096-th root of unity 7^((r-1)/4096) of the deneb polynomial-commitments spec, Montgomery form
#define B200_FR_OMEGA_4096 {{0x09458a39u, 0xf2df262cu, 0x99dff177u, 0x048cdf5bu, 0xc7cce57bu, 0x16857bc5u, 0xa4a915aeu, 0x043b3dbcu}}
// 1/4096 mod r, Montgomery form (= 2^244)
#define B200_FR_INV_4096 {{0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00100000u}}

B200_HD Fr fr_r() { Fr r = B200_FR_R; return r; }
B200_HD Fr fr_zero() { Fr r = {{0, 0, 0, 0, 0, 0, 0, 0}}; return r; }
B200_HD Fr fr_one() { Fr r = B200_FR_ONE; return r; }

B200_HD bool fr_is_zero(const Fr& a) {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) acc |= a.l[i];
    return acc == 0;
}
B200_HD bool fr_eq(const Fr& a, const Fr& b) {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) acc |= a.l[i] ^ b.l[i];
    return acc == 0;
}
// a < r as a 256-bit integer: the canonical check of a decoded field element
B200_HD bool fr_is_canonical(const Fr& a) {
    const Fr r = fr_r();
    uint64_t borrow = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) borrow = ((uint64_t(a.l[i]) - r.l[i] - borrow) >> 32) & 1;
    return borrow != 0;
}

// raw 256-bit add / subtract: hardware carry chains on the device (one IADD3.X per limb), 64-bit emulation on the host
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ uint32_t fr_add_raw(Fr& r, const Fr& a, const Fr& b) {
    uint32_t c;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7]), "=r"(c)
        : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]),
          "r"(b.l[0]), "r"(b.l[1]), "r"(b.l[2]), "r"(b.l[3]), "r"(b.l[4]), "r"(b.l[5]), "r"(b.l[6]), "r"(b.l[7]));
    return c;
}
__device__ __forceinline__ uint32_t fr_sub_raw(Fr& r, const Fr& a, const Fr& b) {
    uint32_t c;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7]), "=r"(c)
        : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]),
          "r"(b.l[0]), "r"(b.l[1]), "r"(b.l[2]), "r"(b.l[3]), "r"(b.l[4]), "r"(b.l[5]), "r"(b.l[6]), "r"(b.l[7]));
    return c & 1u;
}
#else
B200_HD uint32_t fr_add_raw(Fr& r, const Fr& a, const Fr& b) {
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += uint64_t(a.l[i]) + b.l[i]; r.l[i] = uint32_t(c); c >>= 32; }
    return uint32_t(c);
}
B200_HD uint32_t fr_sub_raw(Fr& r, const Fr& a, const Fr& b) {
    uint64_t borrow = 0;
    for (int i = 0; i < 8; i++) {
        const uint64_t d = uint64_t(a.l[i]) - b.l[i] - borrow;
        r.l[i] = uint32_t(d);
        borrow = (d >> 32) & 1;
    }
    return uint32_t(borrow);
}
#endif

// r in [0, 2r) -> [0, r)
B200_HD void fr_reduce_once(Fr& a) {
    const Fr m = fr_r();
    Fr t;
    const uint32_t borrow = fr_sub_raw(t, a, m);
#pragma unroll
    for (int i = 0; i < 8; i++) a.l[i] = borrow ? a.l[i] : t.l[i];
}
B200_HD void fr_add(Fr& r, const Fr& a, const Fr& b) {
    fr_add_raw(r, a, b);   // 2r < 2^256: no carry out
    fr_reduce_once(r);
}
B200_HD void fr_sub(Fr& r, const Fr& a, const Fr& b) {
    Fr t;
    const uint32_t borrow = fr_sub_raw(t, a, b);
    Fr m = fr_r();
#pragma unroll
    for (int i = 0; i < 8; i++) m.l[i] &= 0u - borrow;
    fr_add_raw(r, t, m);
}
B200_HD void fr_neg(Fr& r, const Fr& a) { fr_sub(r, fr_zero(), a); }

// Montgomery product a * b / 2^256 mod r (CIOS, 8 x 8 32x32->64 multiply-adds for the product and as many for the
// reduction).  Inputs < r, output < r.
B200_HD void fr_mul(Fr& out, const Fr& a, const Fr& b) {
    const Fr m = fr_r();
    uint32_t t[10];
#pragma unroll
    for (int j = 0; j < 10; j++) t[j] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t c = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            c += uint64_t(a.l[j]) * b.l[i] + t[j];
            t[j] = uint32_t(c);
            c >>= 32;
        }
        c += t[8];
        t[8] = uint32_t(c);
        t[9] = uint32_t(c >> 32);
        const uint32_t q = t[0] * B200_FR_N0;
        c = (uint64_t(q) * m.l[0] + t[0]) >> 32;
#pragma unroll
        for (int j = 1; j < 8; j++) {
            c += uint64_t(q) * m.l[j] + t[j];
            t[j - 1] = uint32_t(c);
            c >>= 32;
        }
        c += t[8];
        t[7] = uint32_t(c);
        t[8] = t[9] + uint32_t(c >> 32);
    }
    Fr r;
#pragma unroll
    for (int j = 0; j < 8; j++) r.l[j] = t[j];
    fr_reduce_once(r);
    out = r;
}
B200_HD void fr_sqr(Fr& r, const Fr& a) { fr_mul(r, a, a); }

B200_HD void fr_to_mont(Fr& r, const Fr& a) { const Fr r2 = B200_FR_R2; fr_mul(r, a, r2); }
B200_HD void fr_from_mont(Fr& r, const Fr& a) {
    Fr one = fr_zero();
    one.l[0] = 1;
    fr_mul(r, a, one);
}

// r = a^e for a 256-bit exponent given as canonical limbs (square-and-multiply from the top bit)
B200_HD void fr_pow(Fr& r, const Fr& a, const Fr& e) {
    Fr acc = fr_one();
#pragma unroll 1
    for (int bit = 255; bit >= 0; bit--) {
        fr_sqr(acc, acc);
        if ((e.l[bit >> 5] >> (bit & 31)) & 1u) fr_mul(acc, acc, a);
    }
    r = acc;
}
// a^(r-2): the inverse of a non-zero element (0 -> 0)
B200_HD void fr_inv(Fr& r, const Fr& a) {
    Fr e = fr_r();
    e.l[0] = 0xffffffffu;   // r - 2: the low limb of r is 1, so the subtraction borrows from limb 1 (0xffffffff)
    e.l[1] = 0xfffffffeu;
    fr_pow(r, a, e);
}

// 32 big-endian bytes -> raw limbs (no reduction)
B200_HD void fr_from_be32_raw(Fr& r, const uint8_t* b) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint8_t* p = b + 28 - 4 * i;
        r.l[i] = (uint32_t(p[0]) << 24) | (uint32_t(p[1]) << 16) | (uint32_t(p[2]) << 8) | p[3];
    }
}
// bytes_to_bls_field: 32 big-endian bytes -> Montgomery Fr; false if the integer is >= r
B200_HD bool fr_from_be32(Fr& r, const uint8_t* b) {
    Fr raw;
    fr_from_be32_raw(raw, b);
    if (!fr_is_canonical(raw)) return false;
    fr_to_mont(r, raw);
    return true;
}
// hash_to_bls_field: a 256-bit integer (limbs) reduced mod r (2^256 < 3r: at most two subtractions) -> Montgomery Fr
B200_HD void fr_from_u256_reduce(Fr& r, Fr raw) {
    fr_reduce_once(raw);
    fr_reduce_once(raw);
    fr_to_mont(r, raw);
}
// Montgomery Fr -> canonical 32 big-endian bytes
B200_HD void fr_to_be32(uint8_t* b, const Fr& a) {
    Fr raw;
    fr_from_mont(raw, a);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint8_t* p = b + 28 - 4 * i;
        p[0] = uint8_t(raw.l[i] >> 24); p[1] = uint8_t(raw.l[i] >> 16); p[2] = uint8_t(raw.l[i] >> 8); p[3] = uint8_t(raw.l[i]);
    }
}

}  // namespace b200
