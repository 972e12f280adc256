// fr_dev.cuh -- BN254 scalar field (Fr) arithmetic on the device: the constants uploaded at engine creation and the helpers
// every kernel uses (conversion to and from Montgomery form, product, sum, inversion, 256-bit cell loads).
// Included by engine.cu inside its anonymous namespace, after the SHA-256 constant tables.
#pragma once

// Field constants, derived on the host from p at engine creation (fr_host.h) and uploaded here.
struct FrConsts {
  uint64_t p[4];    // modulus
  uint64_t r1[4];   // 2^256 mod p  (Montgomery form of 1)
  uint64_t mu;      // floor(2^317 / p)
  uint32_t mu32;    // floor(2^285 / p)
  uint32_t pad;
  uint64_t ninv;    // -p^-1 mod 2^64 (Montgomery reduction)
};
__constant__ FrConsts c_fr;

// ---------------------------------------------------------------------------------------------------
// Montgomery form of a raw value v < 2^64:  v * 2^256 mod p, by one 64x256 multiply and a Barrett
// reduction with a 64-bit quotient estimate (q_hat in {q-2, q-1, q}; checked exhaustively on edge
// cases in tests/test_gpu_parity.py::test_montgomery_conversion_matches_python_ints).  Replaces halo2curves `Fr::from(u64)` (one full Montgomery multiply).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mont_from_u64(uint64_t v, uint64_t r[4]) {
  const uint64_t R0 = c_fr.r1[0], R1 = c_fr.r1[1], R2 = c_fr.r1[2], R3 = c_fr.r1[3];
  uint64_t p0, p1, p2, p3, p4;
  {
    uint64_t l1 = v * R1, l2 = v * R2, l3 = v * R3;
    uint64_t h0 = __umul64hi(v, R0), h1 = __umul64hi(v, R1), h2 = __umul64hi(v, R2), h3 = __umul64hi(v, R3);
    p0 = v * R0;
    asm("add.cc.u64 %0, %4, %5;\n\t"
        "addc.cc.u64 %1, %6, %7;\n\t"
        "addc.cc.u64 %2, %8, %9;\n\t"
        "addc.u64 %3, %10, 0;"
        : "=l"(p1), "=l"(p2), "=l"(p3), "=l"(p4)
        : "l"(l1), "l"(h0), "l"(l2), "l"(h1), "l"(l3), "l"(h2), "l"(h3));
  }
  // quotient estimate: q = floor( (P >> 254) * mu / 2^63 )
  uint64_t ph = (p3 >> 62) | (p4 << 2);
  uint64_t qh = __umul64hi(ph, c_fr.mu), ql = ph * c_fr.mu;
  uint64_t q = (qh << 1) | (ql >> 63);
  // r = P - q * p  (mod 2^256; the true value is < 3p < 2^256)
  const uint64_t P0 = c_fr.p[0], P1 = c_fr.p[1], P2 = c_fr.p[2], P3 = c_fr.p[3];
  uint64_t m0 = q * P0, m1, m2, m3;
  {
    uint64_t l1 = q * P1, l2 = q * P2, l3 = q * P3;
    uint64_t h0 = __umul64hi(q, P0), h1 = __umul64hi(q, P1), h2 = __umul64hi(q, P2);
    asm("add.cc.u64 %0, %3, %4;\n\t"
        "addc.cc.u64 %1, %5, %6;\n\t"
        "addc.u64 %2, %7, %8;"
        : "=l"(m1), "=l"(m2), "=l"(m3)
        : "l"(l1), "l"(h0), "l"(l2), "l"(h1), "l"(l3), "l"(h2));
  }
  uint64_t r0, r1, r2, r3;
  asm("sub.cc.u64 %0, %4, %8;\n\t"
      "subc.cc.u64 %1, %5, %9;\n\t"
      "subc.cc.u64 %2, %6, %10;\n\t"
      "subc.u64 %3, %7, %11;"
      : "=l"(r0), "=l"(r1), "=l"(r2), "=l"(r3)
      : "l"(p0), "l"(p1), "l"(p2), "l"(p3), "l"(m0), "l"(m1), "l"(m2), "l"(m3));
#pragma unroll
  for (int it = 0; it < 2; it++) {
    uint64_t s0, s1, s2, s3, borrow;
    asm("sub.cc.u64 %0, %5, %9;\n\t"
        "subc.cc.u64 %1, %6, %10;\n\t"
        "subc.cc.u64 %2, %7, %11;\n\t"
        "subc.cc.u64 %3, %8, %12;\n\t"
        "subc.u64 %4, 0, 0;"
        : "=l"(s0), "=l"(s1), "=l"(s2), "=l"(s3), "=l"(borrow)
        : "l"(r0), "l"(r1), "l"(r2), "l"(r3), "l"(P0), "l"(P1), "l"(P2), "l"(P3));
    if (borrow == 0) { r0 = s0; r1 = s1; r2 = s2; r3 = s3; }
  }
  r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3;
}
// p - r (r != 0), 0 for r == 0
__device__ __forceinline__ void fr_negate(uint64_t r[4]) {
  if ((r[0] | r[1] | r[2] | r[3]) == 0) return;
  uint64_t s0, s1, s2, s3;
  asm("sub.cc.u64 %0, %4, %8;\n\t"
      "subc.cc.u64 %1, %5, %9;\n\t"
      "subc.cc.u64 %2, %6, %10;\n\t"
      "subc.u64 %3, %7, %11;"
      : "=l"(s0), "=l"(s1), "=l"(s2), "=l"(s3)
      : "l"(c_fr.p[0]), "l"(c_fr.p[1]), "l"(c_fr.p[2]), "l"(c_fr.p[3]), "l"(r[0]), "l"(r[1]), "l"(r[2]), "l"(r[3]));
  r[0] = s0; r[1] = s1; r[2] = s2; r[3] = s3;
}

// Same conversion for v < 2^32: 32x256 multiply, 32-bit quotient estimate q_hat = ((P >> 254) * floor(2^285/p)) >> 31
// (q_hat in {q-2, q-1, q}), r = P - q_hat * p, two conditional subtractions; carry chains in PTX.
__device__ __forceinline__ void mont_from_u32(uint32_t v, uint32_t x[8]) {
  const uint32_t* R = reinterpret_cast<const uint32_t*>(c_fr.r1);
  const uint32_t* PM = reinterpret_cast<const uint32_t*>(c_fr.p);
  // P = v * R (9 limbs) and M = low 256 bits of q * p, each as one chain of 32x32+64 multiply-adds (IMAD.WIDE: both halves
  // of a product from one instruction, the carry rides in the 64-bit accumulator)
  uint32_t pl[9];
  {
    uint64_t acc = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      acc = (uint64_t)v * R[k] + (acc >> 32);
      pl[k] = (uint32_t)acc;
    }
    pl[8] = (uint32_t)(acc >> 32);
  }
  const uint32_t ph = __funnelshift_r(pl[7], pl[8], 30);   // (P >> 254), < 2^32
  const uint32_t q = (uint32_t)(((uint64_t)ph * c_fr.mu32) >> 31);
  uint32_t m[8], r[8];
  {
    uint64_t acc = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      acc = (uint64_t)q * PM[k] + (acc >> 32);
      m[k] = (uint32_t)acc;
    }
  }
  asm("sub.cc.u32 %0, %8, %16;\n\t"
      "subc.cc.u32 %1, %9, %17;\n\t"
      "subc.cc.u32 %2, %10, %18;\n\t"
      "subc.cc.u32 %3, %11, %19;\n\t"
      "subc.cc.u32 %4, %12, %20;\n\t"
      "subc.cc.u32 %5, %13, %21;\n\t"
      "subc.cc.u32 %6, %14, %22;\n\t"
      "subc.u32 %7, %15, %23;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(pl[0]), "r"(pl[1]), "r"(pl[2]), "r"(pl[3]), "r"(pl[4]), "r"(pl[5]), "r"(pl[6]), "r"(pl[7]),
        "r"(m[0]), "r"(m[1]), "r"(m[2]), "r"(m[3]), "r"(m[4]), "r"(m[5]), "r"(m[6]), "r"(m[7]));
#pragma unroll
  for (int it = 0; it < 2; it++) {
    uint32_t s[8], b;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(s[4]), "=r"(s[5]), "=r"(s[6]), "=r"(s[7]), "=r"(b)
        : "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(PM[0]), "r"(PM[1]), "r"(PM[2]), "r"(PM[3]), "r"(PM[4]), "r"(PM[5]), "r"(PM[6]), "r"(PM[7]));
    if (b == 0) {
#pragma unroll
      for (int k = 0; k < 8; k++) r[k] = s[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 8; k++) x[k] = r[k];
}
__device__ __forceinline__ void fr_negate32(uint32_t x[8]) {
  const uint32_t* PM = reinterpret_cast<const uint32_t*>(c_fr.p);
  uint32_t any = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) any |= x[k];
  if (!any) return;
  uint32_t b = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const uint64_t d = (uint64_t)PM[k] - x[k] - b;
    x[k] = (uint32_t)d;
    b = (uint32_t)(d >> 63);
  }
}

// Montgomery reduction: x * 2^-256 mod p, canonical (Montgomery form -> the integer the cell stands for)
__device__ __forceinline__ void mont_reduce(const uint64_t x[4], uint64_t r[4]) {
  typedef unsigned __int128 u128;
  uint64_t t0 = x[0], t1 = x[1], t2 = x[2], t3 = x[3];
  const uint64_t P0 = c_fr.p[0], P1 = c_fr.p[1], P2 = c_fr.p[2], P3 = c_fr.p[3];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const uint64_t m = t0 * c_fr.ninv;
    u128 c = (u128)m * P0 + t0;            // low limb becomes 0
    c = (u128)m * P1 + t1 + (uint64_t)(c >> 64); t0 = (uint64_t)c;
    c = (u128)m * P2 + t2 + (uint64_t)(c >> 64); t1 = (uint64_t)c;
    c = (u128)m * P3 + t3 + (uint64_t)(c >> 64); t2 = (uint64_t)c;
    t3 = (uint64_t)(c >> 64);
  }
  // t < 2p: one conditional subtraction
  uint64_t s0, s1, s2, s3, borrow;
  asm("sub.cc.u64 %0, %5, %9;\n\t"
      "subc.cc.u64 %1, %6, %10;\n\t"
      "subc.cc.u64 %2, %7, %11;\n\t"
      "subc.cc.u64 %3, %8, %12;\n\t"
      "subc.u64 %4, 0, 0;"
      : "=l"(s0), "=l"(s1), "=l"(s2), "=l"(s3), "=l"(borrow)
      : "l"(t0), "l"(t1), "l"(t2), "l"(t3), "l"(P0), "l"(P1), "l"(P2), "l"(P3));
  if (borrow == 0) { t0 = s0; t1 = s1; t2 = s2; t3 = s3; }
  r[0] = t0; r[1] = t1; r[2] = t2; r[3] = t3;
}

__device__ __forceinline__ void load_cell(const uint64_t* p, uint64_t x[4]) {
  const ulonglong2 a = reinterpret_cast<const ulonglong2*>(p)[0], b = reinterpret_cast<const ulonglong2*>(p)[1];
  x[0] = a.x; x[1] = a.y; x[2] = b.x; x[3] = b.y;
}

// Montgomery product a * b * 2^-256 mod p (CIOS), inputs < p
__device__ __forceinline__ void mont_mul_dev(const uint64_t a[4], const uint64_t b[4], uint64_t r[4]) {
  typedef unsigned __int128 u128;
  const uint64_t P0 = c_fr.p[0], P1 = c_fr.p[1], P2 = c_fr.p[2], P3 = c_fr.p[3];
  uint64_t t0 = 0, t1 = 0, t2 = 0, t3 = 0, t4 = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    u128 c = (u128)a[0] * b[i] + t0; t0 = (uint64_t)c;
    c = (u128)a[1] * b[i] + t1 + (uint64_t)(c >> 64); t1 = (uint64_t)c;
    c = (u128)a[2] * b[i] + t2 + (uint64_t)(c >> 64); t2 = (uint64_t)c;
    c = (u128)a[3] * b[i] + t3 + (uint64_t)(c >> 64); t3 = (uint64_t)c;
    c = (u128)t4 + (uint64_t)(c >> 64);
    t4 = (uint64_t)c;
    const uint64_t t5 = (uint64_t)(c >> 64);
    const uint64_t m = t0 * c_fr.ninv;
    c = (u128)m * P0 + t0;
    c = (u128)m * P1 + t1 + (uint64_t)(c >> 64); t0 = (uint64_t)c;
    c = (u128)m * P2 + t2 + (uint64_t)(c >> 64); t1 = (uint64_t)c;
    c = (u128)m * P3 + t3 + (uint64_t)(c >> 64); t2 = (uint64_t)c;
    c = (u128)t4 + (uint64_t)(c >> 64);
    t3 = (uint64_t)c;
    t4 = t5 + (uint64_t)(c >> 64);
  }
  uint64_t s0, s1, s2, s3, borrow;
  asm("sub.cc.u64 %0, %5, %9;\n\t"
      "subc.cc.u64 %1, %6, %10;\n\t"
      "subc.cc.u64 %2, %7, %11;\n\t"
      "subc.cc.u64 %3, %8, %12;\n\t"
      "subc.u64 %4, %13, 0;"
      : "=l"(s0), "=l"(s1), "=l"(s2), "=l"(s3), "=l"(borrow)
      : "l"(t0), "l"(t1), "l"(t2), "l"(t3), "l"(P0), "l"(P1), "l"(P2), "l"(P3), "l"(t4));
  if ((borrow >> 63) == 0) { t0 = s0; t1 = s1; t2 = s2; t3 = s3; }   // t >= p (t4 carries the 257th bit)
  r[0] = t0; r[1] = t1; r[2] = t2; r[3] = t3;
}

// (x + y) mod p and (x - y) mod p for x, y < p
__device__ __forceinline__ void fr_add_dev(const uint64_t x[4], const uint64_t y[4], uint64_t r[4]) {
  typedef unsigned __int128 u128;
  u128 c = (u128)x[0] + y[0]; uint64_t t0 = (uint64_t)c;
  c = (u128)x[1] + y[1] + (uint64_t)(c >> 64); uint64_t t1 = (uint64_t)c;
  c = (u128)x[2] + y[2] + (uint64_t)(c >> 64); uint64_t t2 = (uint64_t)c;
  c = (u128)x[3] + y[3] + (uint64_t)(c >> 64); uint64_t t3 = (uint64_t)c;   // p < 2^254: no carry out
  uint64_t s0, s1, s2, s3, borrow;
  asm("sub.cc.u64 %0, %5, %9;\n\t"
      "subc.cc.u64 %1, %6, %10;\n\t"
      "subc.cc.u64 %2, %7, %11;\n\t"
      "subc.cc.u64 %3, %8, %12;\n\t"
      "subc.u64 %4, 0, 0;"
      : "=l"(s0), "=l"(s1), "=l"(s2), "=l"(s3), "=l"(borrow)
      : "l"(t0), "l"(t1), "l"(t2), "l"(t3), "l"(c_fr.p[0]), "l"(c_fr.p[1]), "l"(c_fr.p[2]), "l"(c_fr.p[3]));
  if (borrow == 0) { t0 = s0; t1 = s1; t2 = s2; t3 = s3; }
  r[0] = t0; r[1] = t1; r[2] = t2; r[3] = t3;
}

__device__ __forceinline__ void fr_one(uint64_t r[4]) { r[0] = c_fr.r1[0]; r[1] = c_fr.r1[1]; r[2] = c_fr.r1[2]; r[3] = c_fr.r1[3]; }
__device__ __forceinline__ bool fr_is_zero(const uint64_t x[4]) { return (x[0] | x[1] | x[2] | x[3]) == 0; }
__device__ __forceinline__ void fr_copy(const uint64_t x[4], uint64_t r[4]) { r[0] = x[0]; r[1] = x[1]; r[2] = x[2]; r[3] = x[3]; }
__device__ __forceinline__ void fr_mul_into(uint64_t acc[4], const uint64_t x[4]) {
  uint64_t t[4];
  mont_mul_dev(acc, x, t);
  fr_copy(t, acc);
}

// x^(p-2) (Fermat), x != 0; Montgomery in and out
__device__ void fr_inv_dev(const uint64_t x[4], uint64_t r[4]) {
  const uint64_t e[4] = {c_fr.p[0] - 2, c_fr.p[1], c_fr.p[2], c_fr.p[3]};   // p[0] is odd and > 2: no borrow
  fr_one(r);
  for (int b = 253; b >= 0; b--) {   // p < 2^254
    fr_mul_into(r, r);
    if ((e[b >> 6] >> (b & 63)) & 1u) fr_mul_into(r, x);
  }
}
