// SURVEY.md 8(f)3, the part that can be pinned without the ring-proof crate: products of BLS12-381 pairings and the batched KZG
// opening check of a ring-proof verifier (included at the end of vrfs_b200.cu; kernels + their entry points).
//   e(C_i - [v_i] G1, G2) = e(W_i, [tau - z_i] G2)  for i < k, aggregated with caller-supplied coefficients r_i (the
//   transcript's challenges - inputs here, exactly as the ring's row layout is):
//       L = sum_i r_i C_i + sum_i (r_i z_i) W_i - [sum_i r_i v_i] G1,      R = sum_i r_i W_i,
//       accept  <=>  e(L, G2) e(-R, [tau] G2) = 1
//   = one 2-column MSM over the 2k + 1 bases [C | W | G1] (csrc/msm.cuh) + one product of two pairings (csrc/pairing.cuh).
// The prover's side, vrfs_kzg_open_batch: v = p(z) and W = [q(tau)] G1 for q = (p - p(z)) / (X - z), the quotient as a blocked
// suffix scan (csrc/kzg_open.cuh) and W as the prepared MSM of its coefficients over the monomial SRS.  vrfs_kzg_open_aggregated_batch:
// every p_i(z_g) by chunked evaluation, P_g = sum nu_i p_i per group, and the openings of the P_g through the same slice loop.
#pragma once
#include "kzg_open.cuh"
#ifndef VRFS_PAIRING_LANES_MAX_N
#define VRFS_PAIRING_LANES_MAX_N 4096      // measured cross-over with the one-thread kernel (tools/pairing_bench.py): 4096 products 20 ms vs 27.5 ms
#endif

// one thread per product of `pairs` pairings (tests, small batches, and the reference point for the cooperative kernel)
__global__ void __launch_bounds__(32) k_pairing_products(uint32_t n, int pairs, const uint8_t* g1, const uint8_t* g2, const uint32_t* negate,
                                                        uint8_t* out_verdict, uint8_t* out_gt) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fq12 e = f12_one();
  const int v = pairing_product_check_bytes(pairs, g1 + (size_t)96 * pairs * i, g2 + (size_t)192 * pairs * i, negate ? negate[i] : 0u, &e);
  out_verdict[i] = (uint8_t)v;
  if (out_gt) f12_store(out_gt + (size_t)576 * i, e);
}

// scalars of the aggregated check, column-major over the 2k + 1 bases [C_0..C_{k-1} | W_0..W_{k-1} | G1]:
//   column 0: r_i | r_i z_i | (filled by k_kzg_sum)      column 1: 0 | r_i | 0;      prod[i] = r_i v_i
__global__ void __launch_bounds__(128) k_kzg_scalars(uint32_t k, const uint8_t* z, const uint8_t* v, const uint8_t* r, uint8_t* scal, uint32_t* prod) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= k) return;
  const size_t n = 2 * (size_t)k + 1;
  uint32_t raw[8];
  load_le<8>(raw, r + (size_t)32 * i); const Fr255 ri = to_mont<BlsFr>(raw);
  load_le<8>(raw, z + (size_t)32 * i); const Fr255 zi = to_mont<BlsFr>(raw);
  load_le<8>(raw, v + (size_t)32 * i); const Fr255 vi = to_mont<BlsFr>(raw);
  uint32_t out[8];
  from_mont<BlsFr>(out, ri);
  store_le<8>(scal + (size_t)32 * i, out);                        // col 0, C_i
  store_le<8>(scal + (size_t)32 * (n + k + i), out);              // col 1, W_i
  from_mont<BlsFr>(out, ri * zi);
  store_le<8>(scal + (size_t)32 * (k + i), out);                  // col 0, W_i
  for (int j = 0; j < 8; j++) out[j] = 0;
  store_le<8>(scal + (size_t)32 * (n + i), out);                  // col 1, C_i
  const Fr255 p = ri * vi;
  for (int j = 0; j < 8; j++) prod[(size_t)8 * i + j] = p.v[j];
}
// one block: col 0 of the G1 row = - sum_i r_i v_i; col 1 of it = 0
__global__ void __launch_bounds__(256) k_kzg_sum(uint32_t k, const uint32_t* prod, uint8_t* scal) {
  __shared__ uint32_t sh[256][8];
  Fr255 acc = Fr255::zero();
  for (uint32_t i = threadIdx.x; i < k; i += 256) { Fr255 p; for (int j = 0; j < 8; j++) p.v[j] = prod[(size_t)8 * i + j]; acc = acc + p; }
  for (int j = 0; j < 8; j++) sh[threadIdx.x][j] = acc.v[j];
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) {
      Fr255 a, b;
      for (int j = 0; j < 8; j++) { a.v[j] = sh[threadIdx.x][j]; b.v[j] = sh[threadIdx.x + s][j]; }
      a = a + b;
      for (int j = 0; j < 8; j++) sh[threadIdx.x][j] = a.v[j];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    Fr255 t; for (int j = 0; j < 8; j++) t.v[j] = sh[0][j];
    uint32_t out[8];
    from_mont<BlsFr>(out, neg(t));
    const size_t n = 2 * (size_t)k + 1;
    store_le<8>(scal + (size_t)32 * (2 * (size_t)k), out);
    for (int j = 0; j < 8; j++) out[j] = 0;
    store_le<8>(scal + (size_t)32 * (n + 2 * (size_t)k), out);
  }
}
// what CanonicalDeserialize checks of a G1 point: canonical coordinates, on the curve, (level 2) in the prime-order subgroup
__global__ void __launch_bounds__(128) k_g1_validate(uint32_t n, const uint8_t* pts, int level, uint32_t* bad_count) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1AffPt p;
  bool ok = g1_load_bytes(p, pts + (size_t)96 * i) && g1_on_curve_pt(p);
  if (ok && level >= 2 && !p.inf) ok = g1_in_subgroup(p.x, p.y);
  if (!ok) atomicAdd(bad_count, 1u);
}
// the final product of two pairings of the KZG check, e(L, G2) e(-R, [tau] G2): verdict 1 / 0, or 2 when the MSM inputs were
// malformed.  One warp runs the lane programs of csrc/pairing_coop.cuh (1.x ms; the one-thread form took 27 ms).
static vrfs_status kzg_pairing_launch(vrfs_ctx* ctx, const uint8_t* d_lr, const uint8_t* d_g2s, const uint32_t* d_bad, uint32_t* d_negmask, uint8_t* d_verdict) {
  static_assert(PairingProg::NPAIRS == 2, "the KZG check is a product of two pairings");
  static const uint32_t two = 2u;                    // negate the second G1 point
  CU(cudaMemcpyAsync(d_negmask, &two, 4, cudaMemcpyHostToDevice, ctx->stream));
  k_pairing_products_lanes<<<1, PairingProg::LANES, 0, ctx->stream>>>(1u, d_lr, d_g2s, d_negmask, d_bad, d_verdict, nullptr);
  LAUNCHED_AS(ctx, "kzg_pairing");
  return VRFS_OK;
}

extern "C" vrfs_status vrfs_pairing_product_batch(vrfs_ctx* ctx, size_t n, int n_pairs, const uint8_t* g1, const uint8_t* g2, const uint32_t* negate_masks,
                                                  uint8_t* out_ok, uint8_t* out_gt) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (n_pairs < 1 || n_pairs > PAIRING_MAX_PAIRS || !g1 || !g2 || !out_ok) return fail(ctx, VRFS_BAD_ARG, "bad argument (1 <= n_pairs <= %d, non-null buffers)", PAIRING_MAX_PAIRS);
  ST(begin_call(ctx, n));
  const uint8_t *d_g1, *d_g2, *d_neg = nullptr; uint8_t *d_ok, *d_gt = nullptr;
  ST(stage_in(ctx, BUF_IN0, g1, n * 96 * (size_t)n_pairs, &d_g1)); ST(stage_in(ctx, BUF_IN1, g2, n * 192 * (size_t)n_pairs, &d_g2));
  if (negate_masks) ST(stage_in(ctx, BUF_IN2, negate_masks, n * 4, &d_neg));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_gt) ST(stage_out(ctx, BUF_OUT1, n * 576, &d_gt));
  // few products of two pairings: one WARP per product (csrc/pairing_coop.cuh, ~20x lower latency); large batches keep the
  // one-thread-per-product form, whose throughput is higher once every multiplier pipe has its own products
  if (n_pairs == PairingProg::NPAIRS && n <= VRFS_PAIRING_LANES_MAX_N) {
    k_pairing_products_lanes<<<(unsigned)n, PairingProg::LANES, 0, ctx->stream>>>((uint32_t)n, d_g1, d_g2, (const uint32_t*)d_neg, nullptr, d_ok, d_gt);
    LAUNCHED_AS(ctx, "pairing_products_lanes");
  } else {
    k_pairing_products<<<(unsigned)((n + 31) / 32), 32, 0, ctx->stream>>>((uint32_t)n, n_pairs, d_g1, d_g2, (const uint32_t*)d_neg, d_ok, d_gt);
    LAUNCHED_AS(ctx, "pairing_products");
  }
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_gt) ST(copy_out(ctx, out_gt, d_gt, n * 576));
  return finish_call(ctx);
}

extern "C" vrfs_status vrfs_kzg_batch_verify(vrfs_ctx* ctx, size_t k, const uint8_t* commitments, const uint8_t* points_z, const uint8_t* values_v,
                                             const uint8_t* proofs, const uint8_t* coeffs_r, const uint8_t* g2, const uint8_t* tau_g2, int check_points,
                                             uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (!out_ok || !g2 || !tau_g2 || (k && (!commitments || !points_z || !values_v || !proofs || !coeffs_r))) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (k == 0) { *out_ok = 1; return VRFS_OK; }                   // nothing to check
  if (k > (1u << 24)) return fail(ctx, VRFS_BAD_ARG, "more than 2^24 openings per call are not supported");
  ST(begin_call(ctx, k));
  const size_t n = 2 * k + 1;
  // bases [C | W | G1] as ABI bytes, then Montgomery affine records for the MSM
  void *d_bases = nullptr, *d_scal = nullptr, *d_prod = nullptr, *d_aff = nullptr, *d_g2s = nullptr, *d_misc = nullptr;
  ST(ensure(ctx, BUF_IN0, n * 96, &d_bases));
  ST(ensure(ctx, BUF_IN1, 2 * n * 32, &d_scal));
  ST(ensure(ctx, BUF_X0, k * 32, &d_prod));
  ST(ensure(ctx, BUF_W0, n * sizeof(G1Aff), &d_aff));
  ST(ensure(ctx, BUF_X1, 2 * 192, &d_g2s));
  ST(ensure(ctx, BUF_X2, 64, &d_misc));                           // bad-point counter
  const uint8_t *d_z, *d_v, *d_r; uint8_t *d_lr, *d_ok;
  CU(cudaMemcpyAsync(d_bases, commitments, k * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync((uint8_t*)d_bases + k * 96, proofs, k * 96, cudaMemcpyHostToDevice, ctx->stream));
  static const uint8_t g1_gen[96] = {   // the generator of G1, x | y little-endian
      0xbb, 0xc6, 0x22, 0xdb, 0x0a, 0xf0, 0x3a, 0xfb, 0xef, 0x1a, 0x7a, 0xf9, 0x3f, 0xe8, 0x55, 0x6c, 0x58, 0xac, 0x1b, 0x17, 0x3f, 0x3a, 0x4e, 0xa1, 0x05, 0xb9, 0x74, 0x97, 0x4f, 0x8c, 0x68, 0xc3, 0x0f, 0xac, 0xa9, 0x4f, 0x8c, 0x63, 0x95, 0x26, 0x94, 0xd7, 0x97, 0x31, 0xa7, 0xd3, 0xf1, 0x17, 0xe1, 0xe7, 0xc5, 0x46, 0x29, 0x23, 0xaa, 0x0c, 0xe4, 0x8a, 0x88, 0xa2, 0x44, 0xc7, 0x3c, 0xd0, 0xed, 0xb3, 0x04, 0x2c, 0xcb, 0x18, 0xdb, 0x00, 0xf6, 0x0a, 0xd0, 0xd5, 0x95, 0xe0, 0xf5, 0xfc, 0xe4, 0x8a, 0x1d, 0x74, 0xed, 0x30, 0x9e, 0xa0, 0xf1, 0xa0, 0xaa, 0xe3, 0x81, 0xf4, 0xb3, 0x08};
  CU(cudaMemcpyAsync((uint8_t*)d_bases + 2 * k * 96, g1_gen, 96, cudaMemcpyHostToDevice, ctx->stream));
  ST(stage_in(ctx, BUF_IN2, points_z, k * 32, &d_z)); ST(stage_in(ctx, BUF_IN3, values_v, k * 32, &d_v)); ST(stage_in(ctx, BUF_IN4, coeffs_r, k * 32, &d_r));
  CU(cudaMemcpyAsync(d_g2s, g2, 192, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync((uint8_t*)d_g2s + 192, tau_g2, 192, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemsetAsync(d_misc, 0, 64, ctx->stream));
  ST(stage_out(ctx, BUF_OUT0, 2 * 96, &d_lr)); ST(stage_out(ctx, BUF_OUT1, 16, &d_ok));
  if (check_points) {
    k_g1_validate<<<(unsigned)((2 * k + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)(2 * k), (const uint8_t*)d_bases, check_points, (uint32_t*)d_misc);
    LAUNCHED_AS(ctx, "g1_validate");
  }
  k_kzg_scalars<<<(unsigned)((k + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)k, d_z, d_v, d_r, (uint8_t*)d_scal, (uint32_t*)d_prod);
  LAUNCHED_AS(ctx, "kzg_scalars");
  k_kzg_sum<<<1, 256, 0, ctx->stream>>>((uint32_t)k, (const uint32_t*)d_prod, (uint8_t*)d_scal);
  LAUNCHED_AS(ctx, "kzg_sum");
  k_msm_prep_bases<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, (const uint8_t*)d_bases, (G1Aff*)d_aff);
  LAUNCHED_AS(ctx, "msm_prep_bases");
  ST(msm_stateless_dev(ctx, n, 2, d_aff, (const uint8_t*)d_scal, d_lr, 0));
  ST(kzg_pairing_launch(ctx, d_lr, (const uint8_t*)d_g2s, (const uint32_t*)d_misc, (uint32_t*)d_misc + 8, d_ok));
  ST(copy_out(ctx, out_ok, d_ok, 1));
  return finish_call(ctx);
}

// ---- KZG opening proofs.  One launch of each quotient kernel covers a group of at most 32 polynomials (the MSM's column limit),
// polynomial p of the group is blockIdx.y; its coefficients are the p-th row of len 32-byte LE values, its point zs[p].
// Scan state of a group: agg[p * chunks + c] = A_c, the chunk's value sum_{j in c} a_j z^(j - c CH); carry[..] = K_c, everything
// above chunk c, sum_{j >= (c+1) CH} a_j z^(j - (c+1) CH); seg[(p * chunks + c) * THREADS + t] = the exclusive suffix of segment t
// inside its chunk.
__device__ __forceinline__ Fr255 kzg_load_mont(const uint8_t* p) { return to_mont<BlsFr>(fr_load_reduced(p).v); }
__device__ __forceinline__ Fr255 kzg_coeff(const uint8_t* a, uint32_t len, uint32_t j) { return j < len ? kzg_load_mont(a + (size_t)32 * j) : Fr255::zero(); }
__device__ __forceinline__ KzgSpan kzg_span_shfl_down(const KzgSpan& s, unsigned d) {
  KzgSpan r;
  for (int i = 0; i < 8; i++) { r.h.v[i] = __shfl_down_sync(0xffffffffu, s.h.v[i], d); r.p.v[i] = __shfl_down_sync(0xffffffffu, s.p.v[i], d); }
  return r;
}
// phase 1, grid (chunks, polynomials): segment values, then a block suffix scan (warp shuffles, then the warps above through
// shared memory) gives every segment its exclusive suffix and the chunk its value A_c
__global__ void __launch_bounds__(KZG_OPEN_THREADS) k_kzg_quotient_chunks(uint32_t len, uint32_t chunks, const uint8_t* coeffs, const uint8_t* zs,
                                                                          Fr255* agg, KzgSpan* seg) {
  __shared__ KzgSpan warp_sum[KZG_OPEN_THREADS / 32];
  const uint32_t c = blockIdx.x, p = blockIdx.y, t = threadIdx.x, lane = t & 31u, w = t >> 5;
  const uint8_t* a = coeffs + (size_t)32 * len * p;
  const Fr255 z = kzg_load_mont(zs + (size_t)32 * p);
  const uint32_t base = c * KZG_OPEN_CH + KZG_OPEN_SEG * t;
  KzgSpan s = {kzg_segment_value(z, [&](int m) { return kzg_coeff(a, len, base + m); }), kzg_pow2k(z, KZG_OPEN_LOG_SEG)};
  for (unsigned d = 1; d < 32; d <<= 1) {                        // inclusive suffix over the lanes of the warp
    const KzgSpan up = kzg_span_shfl_down(s, d);
    if (lane + d < 32) s = kzg_span_combine(s, up);
  }
  KzgSpan ex = kzg_span_shfl_down(s, 1);
  if (lane == 31) ex = kzg_span_identity();
  if (lane == 0) warp_sum[w] = s;
  __syncthreads();
  KzgSpan above = kzg_span_identity();
  for (int u = KZG_OPEN_THREADS / 32 - 1; u > (int)w; u--) above = kzg_span_combine(warp_sum[u], above);
  seg[((size_t)p * chunks + c) * KZG_OPEN_THREADS + t] = kzg_span_combine(ex, above);
  if (t == 0) agg[(size_t)p * chunks + c] = kzg_span_combine(s, above).h;
}
// phase 2, one thread per polynomial: K_last = 0, K_c = A_{c+1} + z^CH K_{c+1}
__global__ void __launch_bounds__(32) k_kzg_quotient_carry(uint32_t cols, uint32_t chunks, const uint8_t* zs, const Fr255* agg, Fr255* carry) {
  const uint32_t p = threadIdx.x;
  if (p >= cols) return;
  const KzgSpan step = {Fr255::zero(), kzg_pow2k(kzg_load_mont(zs + (size_t)32 * p), KZG_OPEN_LOG_CH)};
  const Fr255* A = agg + (size_t)p * chunks;
  Fr255* K = carry + (size_t)p * chunks;
  Fr255 k = Fr255::zero();
  K[chunks - 1] = k;
  for (uint32_t c = chunks - 1; c-- > 0;) {
    KzgSpan e = step;
    e.h = A[c + 1];
    K[c] = k = kzg_carry_in(e, k);
  }
}
// phase 3, grid (ceil(n / CH), polynomials): q_i as canonical LE into row i of the polynomial's MSM column (n rows; zeros from
// len - 1 on, chunks above the coefficients included); the thread of coefficient 0 writes v = p(z)
__global__ void __launch_bounds__(KZG_OPEN_THREADS) k_kzg_quotient_finish(uint32_t n, uint32_t len, uint32_t chunks, const uint8_t* coeffs, const uint8_t* zs,
                                                                          const KzgSpan* seg, const Fr255* carry, uint8_t* columns, uint8_t* values) {
  const uint32_t c = blockIdx.x, p = blockIdx.y, t = threadIdx.x;
  const uint32_t base = c * KZG_OPEN_CH + KZG_OPEN_SEG * t;
  uint8_t* col = columns + (size_t)32 * n * p;
  auto store = [&](int m, const Fr255& q) {
    if (base + m >= n) return;
    Fr255 out;
    from_mont<BlsFr>(out.v, q);
    fr_store16(col + (size_t)32 * (base + m), out);
  };
  if (c >= chunks) {                                             // above every coefficient of the polynomial
    for (int m = 0; m < KZG_OPEN_SEG; m++) store(m, Fr255::zero());
    return;
  }
  const uint8_t* a = coeffs + (size_t)32 * len * p;
  const Fr255 z = kzg_load_mont(zs + (size_t)32 * p);
  const Fr255 in = kzg_carry_in(seg[((size_t)p * chunks + c) * KZG_OPEN_THREADS + t], carry[(size_t)p * chunks + c]);
  const Fr255 v = kzg_segment_finish(z, in, [&](int m) { return kzg_coeff(a, len, base + m); }, store);
  if (base == 0) {
    Fr255 out;
    from_mont<BlsFr>(out.v, v);
    fr_store16(values + (size_t)32 * p, out);
  }
}

// evaluation of vrfs_kzg_open_aggregated_batch, grid (every chunk of every polynomial): the polynomials are concatenated
// (coeff_off: n_polys + 1 coefficient offsets), chunk b is chunk b - chunk_off[p] of polynomial p = chunk_poly[b], whose point is
// zs[poly_group[p]].  Segment values, then an ordered reduction of their spans (shuffles in lane order, then the warps in order)
// gives the chunk's value A_b = sum_{j in the chunk} a_j z^(j - its lowest index).
__global__ void __launch_bounds__(KZG_OPEN_THREADS) k_kzg_eval_chunks(const uint8_t* coeffs, const uint64_t* coeff_off, const uint32_t* chunk_off,
                                                                      const uint32_t* chunk_poly, const uint32_t* poly_group, const uint8_t* zs, Fr255* agg) {
  __shared__ KzgSpan warp_sum[KZG_OPEN_THREADS / 32];
  const uint32_t b = blockIdx.x, p = chunk_poly[b], t = threadIdx.x, lane = t & 31u, w = t >> 5;
  const uint64_t off = coeff_off[p];
  const uint32_t len = (uint32_t)(coeff_off[p + 1] - off);
  const uint8_t* a = coeffs + 32 * off;
  const Fr255 z = kzg_load_mont(zs + (size_t)32 * poly_group[p]);
  const uint32_t base = (b - chunk_off[p]) * KZG_OPEN_CH + KZG_OPEN_SEG * t;
  KzgSpan s = {kzg_segment_value(z, [&](int m) { return kzg_coeff(a, len, base + m); }), kzg_pow2k(z, KZG_OPEN_LOG_SEG)};
  // after step d, a lane l with l % 2d = 0 holds the lanes l .. l + 2d - 1 in order (the other lanes' values are never read)
  for (unsigned d = 1; d < 32; d <<= 1) s = kzg_span_combine(s, kzg_span_shfl_down(s, d));
  if (lane == 0) warp_sum[w] = s;
  __syncthreads();
  if (t == 0) {
    KzgSpan c = warp_sum[0];
    for (int u = 1; u < KZG_OPEN_THREADS / 32; u++) c = kzg_span_combine(c, warp_sum[u]);
    agg[b] = c.h;
  }
}
// one thread per polynomial: v_i = sum_c A_c (z^CH)^c over its chunks, canonical LE (0 for a polynomial without coefficients)
__global__ void __launch_bounds__(128) k_kzg_eval_finish(uint32_t n_polys, const uint32_t* chunk_off, const uint32_t* poly_group, const uint8_t* zs,
                                                         const Fr255* agg, uint8_t* values) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_polys) return;
  const Fr255 z_ch = kzg_pow2k(kzg_load_mont(zs + (size_t)32 * poly_group[i]), KZG_OPEN_LOG_CH);
  const Fr255* A = agg + chunk_off[i];
  const Fr255 v = kzg_chunk_horner(z_ch, chunk_off[i + 1] - chunk_off[i], [&](uint32_t c) { return A[c]; });
  Fr255 out;
  from_mont<BlsFr>(out.v, v);
  fr_store16(values + (size_t)32 * i, out);
}
// aggregation, grid (ceil(len / CH), groups of a slice): row j of slice group y (group g0 + y, polynomials group_off[g] ..
// group_off[g + 1] - 1) = sum_{i in the group, j < len_i} nu_i a_{i,j}, canonical LE, rows of len coefficients per group
__global__ void __launch_bounds__(KZG_OPEN_THREADS) k_kzg_aggregate(uint32_t g0, uint32_t len, const uint8_t* coeffs, const uint64_t* coeff_off,
                                                                    const uint32_t* group_off, const uint8_t* nus, uint8_t* out) {
  const uint32_t g = g0 + blockIdx.y, base = blockIdx.x * KZG_OPEN_CH + KZG_OPEN_SEG * threadIdx.x;
  if (base >= len) return;
  Fr255 acc[KZG_OPEN_SEG];
  for (int m = 0; m < KZG_OPEN_SEG; m++) acc[m] = Fr255::zero();
  for (uint32_t i = group_off[g]; i < group_off[g + 1]; i++) {
    const uint64_t off = coeff_off[i];
    const uint32_t len_i = (uint32_t)(coeff_off[i + 1] - off);
    if (base >= len_i) continue;
    const Fr255 nu = kzg_load_mont(nus + (size_t)32 * i);
    const uint8_t* a = coeffs + 32 * (off + base);
    for (int m = 0; m < KZG_OPEN_SEG; m++)
      if (base + m < len_i) acc[m] = acc[m] + kzg_agg_term(nu, fr_load_reduced(a + 32 * m));
  }
  uint8_t* row = out + (size_t)32 * len * blockIdx.y;
  for (int m = 0; m < KZG_OPEN_SEG; m++)
    if (base + m < len) fr_store16(row + (size_t)32 * (base + m), acc[m]);
}

// The opening loop of vrfs_kzg_open_batch and vrfs_kzg_open_aggregated_batch: k polynomials at the points d_z (k * 32 bytes), in
// slices of at most 32 (the MSM's column limit) through the three quotient kernels and the prepared MSM, values and proofs copied
// out slice by slice (values only when out_values is not null).  slice(i0, cols, &a, &len) enqueues whatever produces the
// coefficients of polynomials i0 .. i0 + cols - 1 and names them: cols rows of len <= max_len coefficients on the device.
// Every buffer here is sized for the largest slice before the first one (ensure() may move a buffer, and earlier slices still
// read theirs); the caller sizes its own buffers before calling.
template <class Slice>
static vrfs_status kzg_open_slices(vrfs_ctx* ctx, const vrfs_msm_bases* srs, size_t k, size_t max_len, const uint8_t* d_z, uint8_t* out_values,
                                   uint8_t* out_proofs, Slice slice) {
  const size_t n = srs->n, group = k < 32 ? k : 32, max_chunks = max_len ? (max_len + KZG_OPEN_CH - 1) / KZG_OPEN_CH : 1;
  uint8_t *d_w, *d_v; void *d_cols = nullptr, *d_scan = nullptr;
  ST(ensure(ctx, BUF_X0, group * n * 32, &d_cols));
  ST(ensure(ctx, BUF_X1, group * max_chunks * (2 * sizeof(Fr255) + KZG_OPEN_THREADS * sizeof(KzgSpan)), &d_scan));
  ST(stage_out(ctx, BUF_OUT0, group * 96, &d_w)); ST(stage_out(ctx, BUF_OUT1, group * 32, &d_v));
  for (size_t i0 = 0; i0 < k; i0 += group) {
    const size_t cols = k - i0 < group ? k - i0 : group;
    const uint8_t* a = nullptr; size_t len = 0;
    ST(slice(i0, cols, &a, &len));
    const size_t chunks = len ? (len + KZG_OPEN_CH - 1) / KZG_OPEN_CH : 1;
    Fr255* agg = (Fr255*)d_scan;
    Fr255* carry = agg + group * chunks;
    KzgSpan* seg = (KzgSpan*)(carry + group * chunks);
    const uint8_t* z = d_z + 32 * i0;
    k_kzg_quotient_chunks<<<dim3((unsigned)chunks, (unsigned)cols), KZG_OPEN_THREADS, 0, ctx->stream>>>((uint32_t)len, (uint32_t)chunks, a, z, agg, seg);
    LAUNCHED_AS(ctx, "kzg_quotient_chunks");
    k_kzg_quotient_carry<<<1, 32, 0, ctx->stream>>>((uint32_t)cols, (uint32_t)chunks, z, agg, carry);
    LAUNCHED_AS(ctx, "kzg_quotient_carry");
    k_kzg_quotient_finish<<<dim3((unsigned)((n + KZG_OPEN_CH - 1) / KZG_OPEN_CH), (unsigned)cols), KZG_OPEN_THREADS, 0, ctx->stream>>>(
        (uint32_t)n, (uint32_t)len, (uint32_t)chunks, a, z, seg, carry, (uint8_t*)d_cols, d_v);
    LAUNCHED_AS(ctx, "kzg_quotient_finish");
    if (len > 1) ST(msm_prepared_dev(ctx, srs, (int)cols, 0, (const uint8_t*)d_cols, d_w, 0));
    else CU(cudaMemsetAsync(d_w, 0, cols * 96, ctx->stream));  // q = 0: every proof is the identity
    if (out_values) ST(copy_out(ctx, out_values + 32 * i0, d_v, cols * 32));
    ST(copy_out(ctx, out_proofs + 96 * i0, d_w, cols * 96));
  }
  return VRFS_OK;
}

#define KZG_OPEN_MAX_COEFFS (1ull << 26)
extern "C" vrfs_status vrfs_kzg_open_batch(vrfs_ctx* ctx, const vrfs_msm_bases* srs, size_t k, size_t len, const uint8_t* coeffs, const uint8_t* points_z,
                                           uint8_t* out_values, uint8_t* out_proofs) {
  if (!ctx || !srs || srs->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (k == 0) return VRFS_OK;
  if (!coeffs || !points_z || !out_values || !out_proofs) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (len > srs->n) return fail(ctx, VRFS_BAD_ARG, "polynomial longer than the SRS (len %zu > n %zu)", len, srs->n);
  if (k > KZG_OPEN_MAX_COEFFS / (len ? len : 1)) return fail(ctx, VRFS_BAD_ARG, "more than 2^26 coefficients per call are not supported");
  ST(begin_call(ctx, k));
  const uint8_t *d_a, *d_z;
  ST(stage_in(ctx, BUF_IN0, coeffs, k * len * 32, &d_a)); ST(stage_in(ctx, BUF_IN1, points_z, k * 32, &d_z));
  ST(kzg_open_slices(ctx, srs, k, len, d_z, out_values, out_proofs, [&](size_t i0, size_t, const uint8_t** a, size_t* l) {
    *a = d_a + 32 * len * i0; *l = len;
    return VRFS_OK;
  }));
  return finish_call(ctx);
}

#define KZG_OPEN_MAX_POLYS (1u << 16)
extern "C" vrfs_status vrfs_kzg_open_aggregated_batch(vrfs_ctx* ctx, const vrfs_msm_bases* srs, size_t n_groups, size_t n_polys, const uint64_t* group_off,
                                                      const uint64_t* coeff_off, const uint8_t* coeffs, const uint8_t* points_z, const uint8_t* nus,
                                                      uint8_t* out_values, uint8_t* out_agg_values, uint8_t* out_proofs) {
  if (!ctx || !srs || srs->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n_groups > KZG_OPEN_MAX_POLYS || n_polys > KZG_OPEN_MAX_POLYS) return fail(ctx, VRFS_BAD_ARG, "more than 2^16 groups or polynomials per call are not supported");
  if (n_groups == 0) return n_polys ? fail(ctx, VRFS_BAD_ARG, "polynomials without a group (n_groups = 0, n_polys = %zu)", n_polys) : VRFS_OK;
  if (!group_off || !coeff_off || !points_z || !out_proofs || (n_polys && (!nus || !out_values))) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (group_off[0] != 0 || group_off[n_groups] != n_polys) return fail(ctx, VRFS_BAD_ARG, "group offsets must run from 0 to n_polys");
  for (size_t g = 0; g < n_groups; g++) if (group_off[g + 1] < group_off[g]) return fail(ctx, VRFS_BAD_ARG, "group offsets must be non-decreasing");
  if (coeff_off[0] != 0) return fail(ctx, VRFS_BAD_ARG, "coefficient offsets must start at 0");
  size_t n_chunks = 0;
  for (size_t i = 0; i < n_polys; i++) {
    if (coeff_off[i + 1] < coeff_off[i]) return fail(ctx, VRFS_BAD_ARG, "coefficient offsets must be non-decreasing");
    const size_t len = coeff_off[i + 1] - coeff_off[i];
    if (len > srs->n) return fail(ctx, VRFS_BAD_ARG, "polynomial %zu longer than the SRS (len %zu > n %zu)", i, len, srs->n);
    n_chunks += (len + KZG_OPEN_CH - 1) / KZG_OPEN_CH;
  }
  const size_t total = coeff_off[n_polys];
  if (total > KZG_OPEN_MAX_COEFFS) return fail(ctx, VRFS_BAD_ARG, "more than 2^26 coefficients per call are not supported");
  if (total && !coeffs) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, n_groups));
  // host-built index tables, one u32 array: chunk_off (n_polys + 1) | poly_group (n_polys) | group_off (n_groups + 1) | chunk_poly (n_chunks)
  std::vector<uint32_t> tab(2 * n_polys + n_groups + 2 + n_chunks);
  uint32_t *chunk_off = tab.data(), *poly_group = chunk_off + n_polys + 1, *goff = poly_group + n_polys, *chunk_poly = goff + n_groups + 1;
  std::vector<size_t> group_len(n_groups, 0);      // the longest polynomial of each group
  chunk_off[0] = 0;
  for (size_t g = 0; g < n_groups; g++) {
    goff[g] = (uint32_t)group_off[g];
    for (uint64_t i = group_off[g]; i < group_off[g + 1]; i++) {
      const size_t len = coeff_off[i + 1] - coeff_off[i];
      poly_group[i] = (uint32_t)g;
      chunk_off[i + 1] = chunk_off[i] + (uint32_t)((len + KZG_OPEN_CH - 1) / KZG_OPEN_CH);
      for (uint32_t b = chunk_off[i]; b < chunk_off[i + 1]; b++) chunk_poly[b] = (uint32_t)i;
      if (len > group_len[g]) group_len[g] = len;
    }
  }
  goff[n_groups] = (uint32_t)n_polys;
  size_t max_len = 0;
  for (size_t g = 0; g < n_groups; g++) if (group_len[g] > max_len) max_len = group_len[g];
  const size_t slice = n_groups < 32 ? n_groups : 32;
  // every buffer of the call sized before the first launch (kzg_open_slices sizes its own before its loop)
  const uint8_t *d_a, *d_z, *d_nu, *d_coff, *d_tab; uint8_t* d_vals; void *d_p = nullptr, *d_A = nullptr;
  ST(stage_in(ctx, BUF_IN0, coeffs, total * 32, &d_a)); ST(stage_in(ctx, BUF_IN1, points_z, n_groups * 32, &d_z));
  ST(stage_in(ctx, BUF_IN2, nus, n_polys * 32, &d_nu)); ST(stage_in(ctx, BUF_IN3, coeff_off, (n_polys + 1) * 8, &d_coff));
  ST(stage_in(ctx, BUF_IN4, tab.data(), tab.size() * 4, &d_tab));
  ST(ensure(ctx, BUF_X2, slice * max_len * 32, &d_p));
  ST(ensure(ctx, BUF_X3, n_chunks * sizeof(Fr255), &d_A));
  ST(stage_out(ctx, BUF_X4, n_polys * 32, &d_vals));
  const uint64_t* dc_off = (const uint64_t*)d_coff;
  const uint32_t *d_chunk_off = (const uint32_t*)d_tab, *d_poly_group = d_chunk_off + n_polys + 1, *d_goff = d_poly_group + n_polys,
                 *d_chunk_poly = d_goff + n_groups + 1;
  if (n_chunks) {
    k_kzg_eval_chunks<<<(unsigned)n_chunks, KZG_OPEN_THREADS, 0, ctx->stream>>>(d_a, dc_off, d_chunk_off, d_chunk_poly, d_poly_group, d_z, (Fr255*)d_A);
    LAUNCHED_AS(ctx, "kzg_eval_chunks");
  }
  if (n_polys) {
    k_kzg_eval_finish<<<(unsigned)((n_polys + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n_polys, d_chunk_off, d_poly_group, d_z, (const Fr255*)d_A, d_vals);
    LAUNCHED_AS(ctx, "kzg_eval_finish");
    ST(copy_out(ctx, out_values, d_vals, n_polys * 32));
  }
  // P_g of a slice of groups into X2, rows of the slice's longest polynomial; then the openings of P_g as vrfs_kzg_open_batch's
  ST(kzg_open_slices(ctx, srs, n_groups, max_len, d_z, out_agg_values, out_proofs, [&](size_t g0, size_t cols, const uint8_t** a, size_t* l) {
    size_t len = 0;
    for (size_t g = g0; g < g0 + cols; g++) if (group_len[g] > len) len = group_len[g];
    if (len) {
      k_kzg_aggregate<<<dim3((unsigned)((len + KZG_OPEN_CH - 1) / KZG_OPEN_CH), (unsigned)cols), KZG_OPEN_THREADS, 0, ctx->stream>>>(
          (uint32_t)g0, (uint32_t)len, d_a, dc_off, d_goff, d_nu, (uint8_t*)d_p);
      LAUNCHED_AS(ctx, "kzg_aggregate");
    }
    *a = (const uint8_t*)d_p; *l = len;
    return VRFS_OK;
  }));
  return finish_call(ctx);
}
