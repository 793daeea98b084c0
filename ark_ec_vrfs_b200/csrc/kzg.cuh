// SURVEY.md 8(f)3, the part that can be pinned without the ring-proof crate: products of BLS12-381 pairings and the batched KZG
// opening check of a ring-proof verifier (included at the end of vrfs_b200.cu; kernels + their entry points).
//   e(C_i - [v_i] G1, G2) = e(W_i, [tau - z_i] G2)  for i < k, aggregated with caller-supplied coefficients r_i (the
//   transcript's challenges - inputs here, exactly as the ring's row layout is):
//       L = sum_i r_i C_i + sum_i (r_i z_i) W_i - [sum_i r_i v_i] G1,      R = sum_i r_i W_i,
//       accept  <=>  e(L, G2) e(-R, [tau] G2) = 1
//   = one 2-column MSM over the 2k + 1 bases [C | W | G1] (csrc/msm.cuh) + one product of two pairings (csrc/pairing.cuh).
#pragma once
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
