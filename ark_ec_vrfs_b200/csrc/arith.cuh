// K1/K2 of SURVEY.md 2.5: N x 32-bit-limb Montgomery prime-field arithmetic held in registers.
//
// Replaces, on the device, what the reference gets from ark-ff's `Fp<MontBackend<_, N>>`
// (the `BaseField<S>` / `ScalarField<S>` aliases re-exported at /root/reference/src/lib.rs:13-17).
// Representation: a*R mod p, R = 2^(32N), limbs little-endian, always fully reduced (< p), so that
// equality is limb equality and canonical bytes are one Montgomery reduction away.
//
// The header is also compilable for the host (HD_INLINE functions with plain-C twins of every PTX
// block) so that tests/host_emul can check the arithmetic without a GPU.  The product never runs it
// on the host: every entry point of the library launches kernels.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define HD_INLINE __device__ __forceinline__
#define HD_NOINLINE static __device__ __noinline__   // free functions
#define HD_NOINLINE_M __device__ __noinline__        // member functions
#define VRFS_CONST_TABLE __device__ __constant__
#define VRFS_GLOBAL_TABLE __device__ const            // per-thread indexed tables: global memory (L1/L2), not the constant bank
#else   // host emulation build (g++, tests only)
#define HD_INLINE inline
#define HD_NOINLINE static
#define HD_NOINLINE_M
#define VRFS_CONST_TABLE static const
#define VRFS_GLOBAL_TABLE static const
#endif

#include "gen/mont_chains.cuh"

namespace vrfs {

// Modulus limbs are compile-time immediates: ptxas emits IMAD.X + IMAD.HI.U32.X for the reduction rows instead of one
// IMAD.WIDE.U32.X - the same number of multiplier passes, no registers spent on the modulus.  (Forcing them into registers
// was measured and rejected in round 1: DESIGN.md "K1".)
// Field parameter packs (generated: gen/field_consts.cuh) provide:
//   static constexpr int N; static constexpr bool FULL (p >= 2^(32N-1)); static constexpr uint32_t NINV;
//   HD_INLINE static uint32_t mod(i), one(i) [R mod p], r2(i), r3(i), pm2(i) [p-2], pm1h(i) [(p-1)/2]
template <class P>
struct alignas(16) Fp {
  static constexpr int N = P::N;
  uint32_t v[N];

  HD_INLINE static Fp zero() { Fp r; for (int i = 0; i < N; i++) r.v[i] = 0; return r; }
  HD_INLINE static Fp one() { Fp r; for (int i = 0; i < N; i++) r.v[i] = P::one(i); return r; }
  HD_INLINE static Fp modulus() { Fp r; for (int i = 0; i < N; i++) r.v[i] = P::mod(i); return r; }
  HD_INLINE static Fp r2() { Fp r; for (int i = 0; i < N; i++) r.v[i] = P::r2(i); return r; }
  HD_INLINE static Fp r3() { Fp r; for (int i = 0; i < N; i++) r.v[i] = P::r3(i); return r; }

  HD_INLINE bool is_zero() const { uint32_t o = 0; for (int i = 0; i < N; i++) o |= v[i]; return o == 0; }
  HD_INLINE bool operator==(const Fp& b) const { uint32_t o = 0; for (int i = 0; i < N; i++) o |= v[i] ^ b.v[i]; return o == 0; }
  HD_INLINE bool operator!=(const Fp& b) const { return !(*this == b); }
};

// raw comparisons on limb arrays --------------------------------------------------------------
template <int N>
HD_INLINE bool limbs_geq(const uint32_t* a, const uint32_t* b) {  // a >= b
  uint32_t t[N];
  return MontChains<N>::sub(t, a, b) == 0;
}

// r = (a >= p) ? a - p : a, also subtracting when `carry` (the 2^(32N) bit) is set
template <class P>
HD_INLINE void cond_sub_p(uint32_t* a, uint32_t carry) {
  constexpr int N = P::N;
  uint32_t t[N], m[N];
  for (int i = 0; i < N; i++) m[i] = P::mod(i);
  uint32_t borrow = MontChains<N>::sub(t, a, m);
  bool take = (carry != 0) | (borrow == 0);
  for (int i = 0; i < N; i++) a[i] = take ? t[i] : a[i];
}

template <class P>
HD_INLINE Fp<P> operator+(const Fp<P>& a, const Fp<P>& b) {
  Fp<P> r;
  uint32_t c = MontChains<P::N>::add(r.v, a.v, b.v);
  cond_sub_p<P>(r.v, P::FULL ? c : 0u);
  return r;
}
template <class P>
HD_INLINE Fp<P> operator-(const Fp<P>& a, const Fp<P>& b) {
  constexpr int N = P::N;
  Fp<P> r;
  uint32_t borrow = MontChains<N>::sub(r.v, a.v, b.v);
  uint32_t m[N], mask = 0u - borrow;
  for (int i = 0; i < N; i++) m[i] = P::mod(i) & mask;
  MontChains<N>::add(r.v, r.v, m);
  return r;
}
template <class P>
HD_INLINE Fp<P> neg(const Fp<P>& a) { return Fp<P>::zero() - a; }
template <class P>
HD_INLINE Fp<P> dbl(const Fp<P>& a) { return a + a; }
template <class P>
HD_INLINE Fp<P> select(bool c, const Fp<P>& a, const Fp<P>& b) {  // c ? a : b
  Fp<P> r;
  for (int i = 0; i < P::N; i++) r.v[i] = c ? a.v[i] : b.v[i];
  return r;
}
template <class P>
HD_INLINE Fp<P> cneg(const Fp<P>& a, bool c) { return select(c, neg(a), a); }

// Reduction rows m*p of the Montgomery product/square.  For p = 1 - 2^32 (mod 2^64) (BLS12-381 Fr: p[0] = 1,
// p[1] = 2^32-1, so NINV = -1 and m = -column0) the lowest limb pair of each chain needs no multiplier:
// m*1 = (0 : m) and m*(2^32-1) = (m - [m != 0] : -m).  With NINV = -1 the row's column value c0 is -m itself, and m and
// m - [m != 0] come out of one borrow chain (MontChains::neg_bm1): no compare, no predicated negation - ptxas issued those as
// IMAD.MOV on the multiplier pipe, which the products keep busy.  VRFS_LOW_SPECIAL=0 keeps the generic rows for comparison.
#ifndef VRFS_LOW_SPECIAL
#define VRFS_LOW_SPECIAL 1
#endif
template <class P> struct RedRows {
  typedef MontChains<P::N> C;
  static constexpr bool SPECIAL = P::LOW_1_FF && VRFS_LOW_SPECIAL;
  static_assert(!SPECIAL || P::NINV == 0xffffffffu, "p = 1 - 2^32 (mod 2^64) has NINV = -1");
  struct M { uint32_t m, nb, bm1; };   // the row multiplier; special rows also -m and m - [m != 0]
  static HD_INLINE M mult(uint32_t c0) {
    M r;
    if (SPECIAL) { r.nb = c0; C::neg_bm1(r.m, r.bm1, c0); }
    else { r.m = c0 * P::NINV; r.nb = r.bm1 = 0u; }
    return r;
  }
  static HD_INLINE void even(uint32_t* acc, uint32_t& top, const uint32_t* mod, const M& m) {
    if (SPECIAL) C::mad_row_lo1(acc, top, mod, m.m); else C::mad_row(acc, top, mod, m.m);
  }
  static HD_INLINE void odd_top(uint32_t* acc, const uint32_t* mod, const M& m) {
    if (SPECIAL) C::mad_row_top_loff(acc, mod + 1, m.m, m.nb, m.bm1); else C::mad_row_top(acc, mod + 1, m.m);
  }
  static HD_INLINE void odd_shift(uint32_t* u, uint32_t& v0, const uint32_t* mod, const M& m) {
    if (SPECIAL) C::shift_mad_row_loff(u, v0, mod + 1, m.m, m.nb, m.bm1); else C::shift_mad_row(u, v0, mod + 1, m.m);
  }
};

// ---- pseudo-Mersenne fields p = 2^(32N-1) - c (2^255 - 19): values are PLAIN residues (the generated constants use the
// representation factor 1, so one() = 1, to_mont/from_mont degenerate to a reduction / a copy), a product is the 2N-limb
// schoolbook product (N^2 wide multiply-accumulates) followed by folding with 2^(32N) = 2c: N more multiply-accumulates
// instead of the N^2 + N of a Montgomery reduction.  t < 2^(64N-1).
template <class P>
HD_INLINE void pm_fold(uint32_t* out, const uint32_t* t) {
  constexpr int N = P::N;
  typedef MontChains<N> C;
  uint32_t v[N], u[N], r[N], addend[N];
  for (int i = 0; i < N; i++) v[i] = t[i];
  C::mul_row(u, t + N + 1, 2u * P::PM_C);         // odd limbs of the high half: u[j] sits at column j+1
  C::mad_row(v, u[N - 1], t + N, 2u * P::PM_C);   // even limbs at columns 0,2,..; the carry out of column N-1 joins column N
  C::merge(u, v);                                  // value = v[0] + (u[0..N-1] << 32)
  r[0] = v[0];
  for (int j = 1; j < N; j++) r[j] = u[j - 1];
  const uint32_t top = (u[N - 1] << 1) | (r[N - 1] >> 31);   // bits at and above 2^(32N-1): at most a few dozen
  r[N - 1] &= 0x7fffffffu;
  addend[0] = top * P::PM_C;
  for (int j = 1; j < N; j++) addend[j] = 0;
  C::add(r, r, addend);                            // < 2^(32N-1) + 2^10
  cond_sub_p<P>(r, 0u);
  for (int i = 0; i < N; i++) out[i] = r[i];
}

// ---- NIST P-256: p = 2^256 - 2^224 + 2^192 + 2^96 - 1.  Plain residues; the 16-limb product is reduced with the FIPS 186
// word identities (2^256 = delta = 2^224 - 2^192 - 2^96 + 1 mod p) as signed 64-bit column sums.  No multiplier instruction at all.
// The sums carry a bias of 5p (-5, +5, +5, -5 at columns 0, 3, 6, 7 and +5 on the overflow word), which makes the overflow k a small
// NON-NEGATIVE number (0 <= k <= 12; 0..9 seen), so that folding it is two plain 32-bit carry chains instead of signed 64-bit columns:
//   r + k delta            = (r + k + k 2^224) - (k 2^96 + k 2^192)          (9 + 6 instructions), overflow ov in {0, 1}, and then
//   t = r + delta; result  = (ov | carry(t)) ? t : r                          - the last fold and the conditional subtraction of p in one
// (ov = 1: r < 2^228, r + delta = value - p < p;  ov = 0: r + delta carries exactly when r >= p, and is r - p then).
// 32 + 9 selects where three signed folds and a conditional subtraction took ~100 instructions.  Checked in Python on all 2^16 products
// with limbs in {0, 2^32 - 1}, 3 * 10^5 random / extreme 512-bit inputs and products near p^2 before this was written.
// r (8 limbs) += k * delta; returns the overflow word
HD_INLINE uint32_t p256_add_k_delta(uint32_t* r, uint32_t k) {
  uint32_t ov;
#ifdef __CUDA_ARCH__
  asm("add.cc.u32 %0, %0, %9; addc.cc.u32 %1, %1, 0; addc.cc.u32 %2, %2, 0; addc.cc.u32 %3, %3, 0; addc.cc.u32 %4, %4, 0; addc.cc.u32 %5, %5, 0; "
      "addc.cc.u32 %6, %6, 0; addc.cc.u32 %7, %7, %9; addc.u32 %8, 0, 0;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(ov) : "r"(k));
  asm("sub.cc.u32 %0, %0, %6; subc.cc.u32 %1, %1, 0; subc.cc.u32 %2, %2, 0; subc.cc.u32 %3, %3, %6; subc.cc.u32 %4, %4, 0; subc.u32 %5, %5, 0;"
      : "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(ov) : "r"(k));
#else
  uint32_t v[9];
  for (int i = 0; i < 8; i++) v[i] = r[i];
  v[8] = 0;
  uint64_t c = 0;
  for (int i = 0; i < 9; i++) { uint64_t t = (uint64_t)v[i] + ((i == 0 || i == 7) ? k : 0u) + c; v[i] = (uint32_t)t; c = t >> 32; }
  uint64_t b = 0;
  for (int i = 0; i < 9; i++) { uint64_t t = (uint64_t)v[i] - ((i == 3 || i == 6) ? k : 0u) - b; v[i] = (uint32_t)t; b = (t >> 32) & 1u; }
  for (int i = 0; i < 8; i++) r[i] = v[i];
  ov = v[8];
#endif
  return ov;
}
template <class P>
HD_INLINE void p256_fold(uint32_t* out, const uint32_t* c) {
  uint32_t r[8], t[8];
  long long a;
#define C64(i) ((long long)c[i])
  a = C64(0) + C64(8) + C64(9) - C64(11) - C64(12) - C64(13) - C64(14) - 5;                      r[0] = (uint32_t)a; a >>= 32;
  a += C64(1) + C64(9) + C64(10) - C64(12) - C64(13) - C64(14) - C64(15);                        r[1] = (uint32_t)a; a >>= 32;
  a += C64(2) + C64(10) + C64(11) - C64(13) - C64(14) - C64(15);                                 r[2] = (uint32_t)a; a >>= 32;
  a += C64(3) + 2 * (C64(11) + C64(12)) + C64(13) - C64(15) - C64(8) - C64(9) + 5;               r[3] = (uint32_t)a; a >>= 32;
  a += C64(4) + 2 * (C64(12) + C64(13)) + C64(14) - C64(9) - C64(10);                            r[4] = (uint32_t)a; a >>= 32;
  a += C64(5) + 2 * (C64(13) + C64(14)) + C64(15) - C64(10) - C64(11);                           r[5] = (uint32_t)a; a >>= 32;
  a += C64(6) + 3 * C64(14) + 2 * C64(15) + C64(13) - C64(8) - C64(9) + 5;                       r[6] = (uint32_t)a; a >>= 32;
  a += C64(7) + 3 * C64(15) + C64(8) - C64(10) - C64(11) - C64(12) - C64(13) - 5;                r[7] = (uint32_t)a; a >>= 32;
#undef C64
  const uint32_t ov = p256_add_k_delta(r, (uint32_t)(a + 5));
  for (int i = 0; i < 8; i++) t[i] = r[i];
  const uint32_t take = ov | p256_add_k_delta(t, 1u);
  for (int i = 0; i < 8; i++) out[i] = take ? t[i] : r[i];
}

// Montgomery product.  Requires a < p; b may be ANY N-limb value (used to reduce hash outputs).
// p < 2^(32N-1): interleaved even/odd accumulators, 2N^2+N multiply-accumulates (IMAD.WIDE.U32).
template <class P>
HD_INLINE void mont_mul_limbs(uint32_t* out, const uint32_t* a, const uint32_t* b) {
  constexpr int N = P::N;
  typedef MontChains<N> C;
  uint32_t mod[N];
  if (P::PM_C != 0) {
    uint32_t t[2 * N];
    C::mul_wide(t, a, b);
    pm_fold<P>(out, t);
  } else if (P::SOLINAS_P256) {
    uint32_t t[2 * N];
    C::mul_wide(t, a, b);
    p256_fold<P>(out, t);
  } else if (!P::FULL) {
    for (int i = 0; i < N; i++) mod[i] = P::mod(i);
    uint32_t u[N], v[N];
    // first row: v = a_even*b0 (cols 0..N-1), u = a_odd*b0 (cols 1..N)
    C::mul_row(v, a, b[0]);
    C::mul_row(u, a + 1, b[0]);
    {
      const typename RedRows<P>::M m = RedRows<P>::mult(v[0]);
      RedRows<P>::odd_top(u, mod, m);
      RedRows<P>::even(v, u[N - 1], mod, m);
    }
#pragma unroll
    for (int i = 1; i < N; i++) {
      if (i & 1) {  // roles: dead-even = v, odd = u
        C::shift_mad_row(v, u[0], a + 1, b[i]);
        C::mad_row(u, v[N - 1], a, b[i]);
        const typename RedRows<P>::M m = RedRows<P>::mult(u[0]);
        RedRows<P>::odd_top(v, mod, m);
        RedRows<P>::even(u, v[N - 1], mod, m);
      } else {
        C::shift_mad_row(u, v[0], a + 1, b[i]);
        C::mad_row(v, u[N - 1], a, b[i]);
        const typename RedRows<P>::M m = RedRows<P>::mult(v[0]);
        RedRows<P>::odd_top(u, mod, m);
        RedRows<P>::even(v, u[N - 1], mod, m);
      }
    }
    // N even: after the last (odd-index) iteration the live odd array is v, the dead-even one is u
    C::merge(v, u);
    cond_sub_p<P>(v, 0u);
    for (int i = 0; i < N; i++) out[i] = v[i];
  } else {
    // p >= 2^(32N-1) (P-256 p and n): textbook CIOS on 64-bit temporaries with the extra top word.
    for (int i = 0; i < N; i++) mod[i] = P::mod(i);
    uint32_t t[N + 2];
    for (int i = 0; i < N + 2; i++) t[i] = 0;
    for (int i = 0; i < N; i++) {
      uint64_t c = 0;
      for (int j = 0; j < N; j++) { uint64_t x = (uint64_t)a[j] * b[i] + t[j] + c; t[j] = (uint32_t)x; c = x >> 32; }
      uint64_t x = (uint64_t)t[N] + c; t[N] = (uint32_t)x; t[N + 1] = (uint32_t)(x >> 32);
      uint32_t m = t[0] * P::NINV;
      x = (uint64_t)m * mod[0] + t[0]; c = x >> 32;
      for (int j = 1; j < N; j++) { x = (uint64_t)m * mod[j] + t[j] + c; t[j - 1] = (uint32_t)x; c = x >> 32; }
      x = (uint64_t)t[N] + c; t[N - 1] = (uint32_t)x; t[N] = t[N + 1] + (uint32_t)(x >> 32);
    }
    cond_sub_p<P>(t, t[N]);
    for (int i = 0; i < N; i++) out[i] = t[i];
  }
}

// The product is a CALLED function (by-value arguments travel in registers under the device ABI), not
// inlined: a point addition inlines 9 of them and the scalar-multiplication loop then no longer fits the
// instruction caches - the first ncu capture of the inlined build showed `stall_no_instruction` as the top
// stall reason by 4x (profiles/r1a_*).  VRFS_INLINE_MUL=1 restores the inlined form for comparison.
#ifndef VRFS_INLINE_MUL
#define VRFS_INLINE_MUL 0
#endif
template <class P>
HD_NOINLINE Fp<P> mont_mul_call(Fp<P> a, Fp<P> b) {
  Fp<P> r;
  mont_mul_limbs<P>(r.v, a.v, b.v);
  return r;
}
template <class P>
HD_INLINE Fp<P> operator*(const Fp<P>& a, const Fp<P>& b) {
#if VRFS_INLINE_MUL
  Fp<P> r;
  mont_mul_limbs<P>(r.v, a.v, b.v);
  return r;
#else
  return mont_mul_call<P>(a, b);
#endif
}
// Montgomery square: the 2N-limb square from N(N+1)/2 wide products (MontChains::sqr_wide), then a reduction-only
// pass of the same even/odd accumulator pair over its low half, then + high half: N(N+1)/2 + N^2 + N multiply-
// accumulates (108 for N = 8) instead of 2N^2 + N (136).  a < p < 2^(32N-1).
#ifndef VRFS_DEDICATED_SQR
#define VRFS_DEDICATED_SQR 1
#endif
// Montgomery reduction of a 2N-limb value t < p * 2^(32N) (a reduction-only pass of the even/odd accumulator pair over the low
// half, then + high half): N^2 + N multiply-accumulates.  Plain Montgomery fields with p < 2^(32N-1) only.
template <class P>
HD_INLINE void mont_reduce_wide(uint32_t* out, const uint32_t* t) {
  constexpr int N = P::N;
  typedef MontChains<N> C;
  uint32_t mod[N], u[N], v[N];
  for (int i = 0; i < N; i++) mod[i] = P::mod(i);
  // reduce the low half: v = even-aligned window (column 0 = v[0]), u = odd-aligned; roles swap every step
  for (int i = 0; i < N; i++) { v[i] = t[i]; u[i] = 0; }
#pragma unroll
  for (int i = 0; i < N; i++) {
    if (i & 1) {   // live-even = u, dead-even (to be shifted) = v
      const typename RedRows<P>::M m = RedRows<P>::mult(u[0] + v[1]);
      RedRows<P>::odd_shift(v, u[0], mod, m);
      RedRows<P>::even(u, v[N - 1], mod, m);
    } else {
      const typename RedRows<P>::M m = RedRows<P>::mult(v[0] + u[1]);
      RedRows<P>::odd_shift(u, v[0], mod, m);
      RedRows<P>::even(v, u[N - 1], mod, m);
    }
  }
  // N even: the last step (odd i) left u as the dead-even array (u[0] = 0) and v as the odd-aligned one
  C::merge(v, u);
  C::add(v, v, t + N);          // + high half: < p + p^2/2^(32N) < 2p < 2^(32N)
  cond_sub_p<P>(v, 0u);
  for (int i = 0; i < N; i++) out[i] = v[i];
}
template <class P>
HD_INLINE void mont_sqr_limbs(uint32_t* out, const uint32_t* a) {
  constexpr int N = P::N;
  typedef MontChains<N> C;
  if ((P::FULL && !P::SOLINAS_P256) || !VRFS_DEDICATED_SQR) { mont_mul_limbs<P>(out, a, a); return; }
  uint32_t t[2 * N];
  if constexpr (P::PM_C != 0) { C::sqr_wide(t, a); pm_fold<P>(out, t); return; }
  else if constexpr (P::SOLINAS_P256) {
    // a may use all 256 bits and sqr_wide needs the top bit clear: a = a' + b 2^255, a^2 = a'^2 + b 2^256 a' + b 2^510
    uint32_t lo[N], add[N];
    const uint32_t mask = 0u - (a[N - 1] >> 31);
    for (int i = 0; i < N; i++) lo[i] = a[i];
    lo[N - 1] &= 0x7fffffffu;
    C::sqr_wide(t, lo);
    for (int i = 0; i < N; i++) add[i] = lo[i] & mask;
    add[N - 1] += mask & 0x40000000u;                 // 2^510 = 2^(256 + 224 + 30); the top limb of a' is below 2^31, so this cannot wrap
    C::add(t + N, t + N, add);                        // a^2 < 2^512: no carry out
    p256_fold<P>(out, t);
    return;
  }
  else {
    C::sqr_wide(t, a);
    mont_reduce_wide<P>(out, t);
  }
}
template <class P>
HD_NOINLINE Fp<P> mont_sqr_call(Fp<P> a) {
  Fp<P> r;
  mont_sqr_limbs<P>(r.v, a.v);
  return r;
}
template <class P>
HD_INLINE Fp<P> sqr(const Fp<P>& a) {
#if VRFS_INLINE_MUL
  Fp<P> r;
  mont_sqr_limbs<P>(r.v, a.v);
  return r;
#else
  return mont_sqr_call<P>(a);
#endif
}

// Two independent products / squares.  (A paired CALLED form that lets ptxas interleave the two carry chains was measured at
// 10.709 vs 10.711 M verifies/s in round 1 - no gain - and removed; the formulas keep issuing their products in independent pairs.)
template <class P> HD_INLINE void mul2(Fp<P>& r0, Fp<P>& r1, const Fp<P>& a, const Fp<P>& b, const Fp<P>& c, const Fp<P>& d) { r0 = a * b; r1 = c * d; }
template <class P> HD_INLINE void sqr2(Fp<P>& r0, Fp<P>& r1, const Fp<P>& a, const Fp<P>& c) { r0 = sqr(a); r1 = sqr(c); }

// canonical limbs (value < 2^(32N), not necessarily < p) -> Montgomery form, reduced
template <class P>
HD_INLINE Fp<P> to_mont(const uint32_t* raw) {
  Fp<P> r, r2 = Fp<P>::r2();
  mont_mul_limbs<P>(r.v, r2.v, raw);
  return r;
}
// Montgomery form -> canonical limbs
template <class P>
HD_INLINE void from_mont(uint32_t* raw, const Fp<P>& a) {
  uint32_t one[P::N];
  one[0] = 1;
  for (int i = 1; i < P::N; i++) one[i] = 0;
  mont_mul_limbs<P>(raw, a.v, one);
}
// (hi * 2^(32N) + lo) mod p, in Montgomery form; hi, lo arbitrary N-limb values
template <class P>
HD_INLINE Fp<P> to_mont_wide(const uint32_t* lo, const uint32_t* hi) {
  Fp<P> a, b, r2 = Fp<P>::r2(), r3 = Fp<P>::r3();
  mont_mul_limbs<P>(a.v, r2.v, lo);
  mont_mul_limbs<P>(b.v, r3.v, hi);
  return a + b;
}

// a^e for a public exponent of the field (E::get<P>(i) = limb i, canonical); MSB-first
// square-and-multiply.  The exponent is the same for every thread, so the branch is warp-uniform.
struct ExpPM2 { template <class P> static HD_INLINE uint32_t get(int i) { return P::pm2(i); } };
struct ExpPM1H { template <class P> static HD_INLINE uint32_t get(int i) { return P::pm1h(i); } };
template <class P, class E>
HD_NOINLINE Fp<P> pow_const(const Fp<P>& a) {
  // 4-bit fixed windows, MSB first: 32N squarings + at most 8N + 14 products (bit-serial square-and-multiply needed
  // ~16N products); the exponent is public, so the table index and the skip of zero windows are warp-uniform
  Fp<P> tbl[16];
  tbl[0] = Fp<P>::one(); tbl[1] = a;
#pragma unroll 1
  for (int i = 2; i < 16; i++) tbl[i] = (i & 1) ? tbl[i - 1] * a : sqr(tbl[i >> 1]);
  Fp<P> acc = Fp<P>::one();
  bool started = false;
#pragma unroll 1
  for (int i = P::N * 8 - 1; i >= 0; i--) {
    const uint32_t d = (E::template get<P>(i >> 3) >> ((i & 7) * 4)) & 15u;
    if (started) { acc = sqr(acc); acc = sqr(acc); acc = sqr(acc); acc = sqr(acc); }
    if (d) { acc = started ? acc * tbl[d] : tbl[d]; started = true; }
  }
  return acc;
}
// Fermat inverse; 0 -> 0 (same convention as the oracle's f_inv)
template <class P>
HD_INLINE Fp<P> inv(const Fp<P>& a) { return pow_const<P, ExpPM2>(a); }
// Euler criterion; true for squares and for 0
template <class P>
HD_INLINE bool is_square(const Fp<P>& a) {
  if (a.is_zero()) return true;
  return pow_const<P, ExpPM1H>(a) == Fp<P>::one();
}

// Jacobi symbol (a/p) of a field element by the binary algorithm (shift / compare / subtract on 8-limb integers, no
// multiplier): 1, -1, or 0 for a = 0.  Works on the stored representation directly: the Montgomery factor 2^(32N) is a
// square, so (aR/p) = (a/p).  ~20 K ALU instructions against ~110 K for an Euler-criterion power; the loop trip count is
// data dependent (lanes of a warp finish within a few per cent of each other).
template <class P>
HD_NOINLINE int jacobi(const Fp<P>& x) {
  constexpr int N = P::N;
  typedef MontChains<N> C;
  uint32_t a[N], n[N], t[N];
  for (int i = 0; i < N; i++) { a[i] = x.v[i]; n[i] = P::mod(i); }
  int sign = 1;
  for (int guard = 0; guard < 64 * N + 8; guard++) {
    uint32_t any = 0;
    for (int i = 0; i < N; i++) any |= a[i];
    if (!any) break;
    // strip the factors of two: (2/n) = -1 iff n = 3, 5 (mod 8)
    while (a[0] == 0) { for (int i = 0; i + 1 < N; i++) a[i] = a[i + 1]; a[N - 1] = 0; }      // 32 = even number of halvings
#if defined(__CUDA_ARCH__)
    const int tz = __ffs((int)a[0]) - 1;
#else
    const int tz = __builtin_ctz(a[0]);
#endif
    if (tz) {
      for (int i = 0; i + 1 < N; i++) a[i] = (a[i] >> tz) | (a[i + 1] << (32 - tz));
      a[N - 1] >>= tz;
      const uint32_t n8 = n[0] & 7u;
      if ((tz & 1) && (n8 == 3u || n8 == 5u)) sign = -sign;
    }
    // both odd now: make a >= n (quadratic reciprocity), then a -= n
    if (C::sub(t, a, n)) {                               // a < n: swap roles, t = n - a
      if ((a[0] & 3u) == 3u && (n[0] & 3u) == 3u) sign = -sign;
      C::sub(t, n, a);
      for (int i = 0; i < N; i++) { n[i] = a[i]; a[i] = t[i]; }
    } else {
      for (int i = 0; i < N; i++) a[i] = t[i];
    }
  }
  uint32_t rest = n[0] ^ 1u;
  for (int i = 1; i < N; i++) rest |= n[i];
  return rest == 0 ? sign : 0;
}

// canonical value > (p-1)/2 ?   (arkworks TE "x is negative" flag, SURVEY A.2)
template <class P>
HD_INLINE bool is_high(const Fp<P>& a) {
  uint32_t raw[P::N], h[P::N], t[P::N];
  from_mont<P>(raw, a);
  for (int i = 0; i < P::N; i++) h[i] = P::pm1h(i);
  return MontChains<P::N>::sub(t, h, raw) != 0;  // borrow <=> raw > (p-1)/2
}
template <class P>
HD_INLINE bool is_odd(const Fp<P>& a) {
  uint32_t raw[P::N];
  from_mont<P>(raw, a);
  return raw[0] & 1u;
}
// is the raw N-limb value canonical (< p)?
template <class P>
HD_INLINE bool is_canonical(const uint32_t* raw) {
  uint32_t m[P::N], t[P::N];
  for (int i = 0; i < P::N; i++) m[i] = P::mod(i);
  return MontChains<P::N>::sub(t, raw, m) != 0;
}

}  // namespace vrfs
