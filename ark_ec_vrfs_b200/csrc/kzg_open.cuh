// The per-thread pieces of the KZG opening quotient (vrfs_kzg_open_batch, kernels in csrc/kzg.cuh).  Host-compilable: the CPU
// tests run them through the same three phases as the kernels (tests/host_emul/hostemu_kzg.cpp), and the evaluation and
// aggregation of vrfs_kzg_open_aggregated_batch likewise (tests/host_emul/hostemu_kzg_agg.cpp).
//   p = sum_{j < len} a_j X^j,  q = (p - p(z)) / (X - z):  q_i = sum_{j > i} a_j z^(j - i - 1),  p(z) = a_0 + z q_0,
// i.e. the suffix recurrence q_{i-1} = a_i + z q_i.  The coefficients, zero-padded at the top, split into chunks of KZG_OPEN_CH
// (one block each), a chunk into segments of KZG_OPEN_SEG (one thread each).  A run of coefficients is a KzgSpan: its value
// as a polynomial in z from its own lowest index, and z^(its length); two adjacent runs combine as lo.h + lo.p * hi.h.
#pragma once
#include "ring.cuh"

namespace vrfs {

#define KZG_OPEN_LOG_SEG 3
#define KZG_OPEN_LOG_THREADS 7
#define KZG_OPEN_SEG (1 << KZG_OPEN_LOG_SEG)                         // coefficients per thread
#define KZG_OPEN_THREADS (1 << KZG_OPEN_LOG_THREADS)                 // threads per chunk (block)
#define KZG_OPEN_LOG_CH (KZG_OPEN_LOG_SEG + KZG_OPEN_LOG_THREADS)
#define KZG_OPEN_CH (1 << KZG_OPEN_LOG_CH)                           // coefficients per chunk

struct KzgSpan { Fr255 h, p; };
HD_INLINE KzgSpan kzg_span_identity() { return {Fr255::zero(), Fr255::one()}; }
HD_INLINE KzgSpan kzg_span_combine(const KzgSpan& lo, const KzgSpan& hi) { return {lo.h + lo.p * hi.h, lo.p * hi.p}; }
// z^(2^e): z^KZG_OPEN_SEG for a segment, z^KZG_OPEN_CH for a chunk
HD_INLINE Fr255 kzg_pow2k(Fr255 z, int e) { for (int i = 0; i < e; i++) z = sqr(z); return z; }

// phase 1, per thread: the value of its segment, sum_m a_{base+m} z^m (ld(m) = a_{base+m} in Montgomery form, zero past len)
template <class Load> HD_INLINE Fr255 kzg_segment_value(const Fr255& z, Load ld) {
  Fr255 h = Fr255::zero();
  for (int m = KZG_OPEN_SEG - 1; m >= 0; m--) h = h * z + ld(m);
  return h;
}
// phase 3, per thread: carry = q_{base+SEG-1} (the exclusive suffix of the chunk above the segment plus z^(distance) times the
// chunk carry, kzg_carry_in); st(m, q) receives q_{base+m}; returns q_{base-1} (p(z) for the segment at index 0)
template <class Load, class Store> HD_INLINE Fr255 kzg_segment_finish(const Fr255& z, const Fr255& carry, Load ld, Store st) {
  Fr255 acc = carry;
  for (int m = KZG_OPEN_SEG - 1; m >= 0; m--) { st(m, acc); acc = acc * z + ld(m); }
  return acc;
}
// suffix above + z^(its distance) * what lies beyond it: the carry into a segment from its chunk (e = the exclusive suffix of the
// segment inside the chunk, k = the chunk's carry K_c), and the chunk carry recurrence K_c = A_{c+1} + z^CH K_{c+1}
HD_INLINE Fr255 kzg_carry_in(const KzgSpan& e, const Fr255& k) { return e.h + e.p * k; }

// vrfs_kzg_open_aggregated_batch.  Evaluation: a chunk's value A_c is the ordered combination of its segments' spans (lower
// segments on the left: kzg_span_combine is not commutative), and p(z) = sum_c A_c (z^CH)^c, by Horner from the top chunk
// (A(c) = A_c, z_ch = z^CH).
template <class Load> HD_INLINE Fr255 kzg_chunk_horner(const Fr255& z_ch, uint32_t chunks, Load A) {
  Fr255 v = Fr255::zero();
  for (uint32_t c = chunks; c-- > 0;) v = v * z_ch + A(c);
  return v;
}
// Aggregation: nu in Montgomery form times a coefficient taken as a plain residue (not converted) is the Montgomery product
// nu a R R^-1 = nu a, again a plain residue; the sums of such terms are the aggregated coefficients, with no conversion either way
HD_INLINE Fr255 kzg_agg_term(const Fr255& nu_mont, const Fr255& a_plain) { return nu_mont * a_plain; }

}  // namespace vrfs
