// K7 + K8 of SURVEY.md 2.5: one item's linear combination
//     R = sum_j  (+/-) k_j * P_j   (variable bases, per item)   +   sum_f (+/-) s_f * B_f  (fixed bases)
// which is every group computation of the hot path (SURVEY.md 3.1-3.3):
//   ietf verify   U = s*G - c*Y            (NV=1, NF=1)      V = s*I - c*O      (NV=2)
//   ietf prove    k*G (NF=1), k*I (NV=1);  Secret::output  sk*I (NV=1);  Public  sk*G (NF=1)
//   pedersen      sk*G + b*B (NF=2), k*G + kb*B (NF=2), k*I, s*I - c*O (NV=2), c*Yb - s*G - sb*B (NV=1, NF=2)
// The reference does each k*P with ark-ec's bit-serial `mul_bigint`; the result is the same group
// element, and every consumer works on its canonical affine encoding.
//
// Variable bases: signed radix-16 fixed windows (no data-dependent branches -> no warp divergence),
// Bandersnatch scalars GLV-split into two 127-bit halves acting on P and psi(P) so a K-term sum costs
// 124 shared doublings + 32*2K additions.  Window tables (9 entries per base incl. the identity)
// live in a per-thread slab of global memory (L2-resident across the resident grid), read with 16-byte loads.
// Fixed bases: signed radix-256 windows over a precomputed table (32-33 x 129 entries, ~400 KB, L2-resident).
// One implementation serves the twisted-Edwards suites (Bandersnatch, Ed25519) and the short-Weierstrass
// one (secp256r1) through the Grp<C> adapter below.
#pragma once
#include "te.cuh"
#include "sw.cuh"
#include "scalar.cuh"

namespace vrfs {

#if !defined(__CUDACC__)
struct uint4 { uint32_t x, y, z, w; };
#endif
#if defined(__CUDACC__)
#define VRFS_HD __host__ __device__
#else
#define VRFS_HD
#endif

template <class F> HD_INLINE void store_fp_xyz(uint32_t* o, const F& X, const F& Y, const F& Z) {   // 3N limbs, 16-byte aligned
  uint4* d = reinterpret_cast<uint4*>(o);
  const uint4 *sx = reinterpret_cast<const uint4*>(X.v), *sy = reinterpret_cast<const uint4*>(Y.v), *sz = reinterpret_cast<const uint4*>(Z.v);
  constexpr int Q = F::N / 4;
  for (int i = 0; i < Q; i++) { d[i] = sx[i]; d[Q + i] = sy[i]; d[2 * Q + i] = sz[i]; }
}
HD_INLINE void prefetch_l2(const void* p, unsigned bytes) {
#ifdef __CUDA_ARCH__
  for (unsigned o = 0; o < bytes; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"((const char*)p + o));
#else
  (void)p; (void)bytes;
#endif
}
HD_INLINE void prefetch_l1(const void* p, unsigned bytes) {
#ifdef __CUDA_ARCH__
  for (unsigned o = 0; o < bytes; o += 128) asm volatile("prefetch.global.L1 [%0];" ::"l"((const char*)p + o));
  if (bytes % 128) asm volatile("prefetch.global.L1 [%0];" ::"l"((const char*)p + bytes - 1));   // entry may straddle two lines
#else
  (void)p; (void)bytes;
#endif
}
template <class T> HD_INLINE void copy_words16(T* dst, const T* src_) {  // sizeof(T) % 16 == 0, both 16-byte aligned
  const uint4* s = reinterpret_cast<const uint4*>(src_);
  uint4* d = reinterpret_cast<uint4*>(dst);
  for (unsigned i = 0; i < sizeof(T) / 16; i++) d[i] = s[i];
}

// ---- group adapters ---------------------------------------------------------------------------
// Fixed-base window width.  16-bit signed windows halve the additions of every fixed-base multiplication (16 instead of 32) at
// the price of a 50 MB table per base (L2/DRAM-resident, prefetched); 8-bit windows keep the tables at 400 KB.
#ifndef VRFS_FIX_BITS
#define VRFS_FIX_BITS 16
#endif
template <class C, bool TE = C::IS_TE> struct Grp;
template <class C> struct Grp<C, true> {
  typedef TEPoint<C> Pt;
  typedef TECached<C> Entry;        // window-table entry
  typedef TEAffCached<C> FixEntry;  // fixed-base table entry
  static constexpr int SPLIT = C::HAS_GLV ? 2 : 1;          // tables per variable base
  static constexpr int WINDOWS = C::HAS_GLV ? 32 : 64;      // radix-16 windows per (half-)scalar
  static constexpr int KB_LIMBS = C::HAS_GLV ? 4 : 8;
  static constexpr int FIX_WINDOWS = 256 / VRFS_FIX_BITS;
  static constexpr int CARRY_WINDOWS = 0;   // r < 2^255: the bias addition never carries out of a 256-bit scalar
  static HD_INLINE void set_identity(Pt& P) { te_set_identity(P); }
  static HD_INLINE void from_affine(Pt& P, const typename C::F& x, const typename C::F& y) { te_from_affine<C>(P, x, y); }
  static HD_INLINE bool on_curve(const typename C::F& x, const typename C::F& y) { return te_on_curve<C>(x, y); }
  static HD_INLINE void to_entry(Entry& e, const Pt& P) { te_to_cached(e, P); }
  // want_t = false: the T coordinate of the sum is left undefined (the caller follows with a doubling, or stores X, Y, Z)
  static HD_INLINE void add_entry(Pt* acc, const Entry* e, bool negate, bool want_t = true) { te_add_cached<C>(acc, acc, e, negate, want_t); }
  static HD_INLINE void add_fix(Pt* acc, const FixEntry* e, bool negate, bool want_t = true) { te_madd<C>(acc, acc, e, negate, want_t); }
  static HD_INLINE void dbl4(Pt* acc) { te_dbl<C>(acc, acc, false); te_dbl<C>(acc, acc, false); te_dbl<C>(acc, acc, false); te_dbl<C>(acc, acc, true); }
  static HD_INLINE void dbl(Pt* acc) { te_dbl<C>(acc, acc, true); }
  static HD_INLINE void dbl_entry(Pt* r, const Entry* e) { Pt p; te_from_cached_xyz<C>(p, *e); te_dbl<C>(r, &p, true); }   // the doubling does not read T
  static HD_INLINE void add(Pt* r, const Pt* p, const Pt* q) { te_add<C>(r, p, q); }
  static HD_INLINE void endo(Pt* r, const Pt* p) { band_endo(reinterpret_cast<TEPoint<BandCurve>*>(r), reinterpret_cast<const TEPoint<BandCurve>*>(p)); }
  static HD_INLINE void to_fix(FixEntry& e, const Pt& P) {
    typename C::F zi = inv(P.Z);
    typename C::F x = P.X * zi, y = P.Y * zi, dt = x * y * C::d();
    if constexpr (C::A_IS_M1) { e.x = y + x; e.y = y - x; e.dt = dt + dt; }       // te.cuh: the a = -1 entry form
    else { e.x = x; e.y = y; e.dt = dt; }
  }
  static HD_INLINE void store_xyz(uint32_t* o, const Pt& P) { store_fp_xyz(o, P.X, P.Y, P.Z); }
  // prepared-key tables: the point (X : Y : Z) (T dropped) back in extended coordinates, and an affine point as a table entry
  static HD_INLINE void from_xyz(Pt& P, const typename C::F& X, const typename C::F& Y, const typename C::F& Z) { P.X = X * Z; P.Y = Y * Z; P.Z = sqr(Z); P.T = X * Y; }
  static HD_INLINE void fix_from_affine(FixEntry& e, const typename C::F& x, const typename C::F& y, bool) {
    typename C::F dt = x * y * C::d();
    if constexpr (C::A_IS_M1) { e.x = y + x; e.y = y - x; e.dt = dt + dt; }
    else { e.x = x; e.y = y; e.dt = dt; }
  }
};
template <class C> struct Grp<C, false> {
  typedef SWPoint<C> Pt;
  typedef SWPoint<C> Entry;
  typedef SWPoint<C> FixEntry;
  static constexpr int SPLIT = 1;
  static constexpr int WINDOWS = 65;       // 64 radix-16 digits + the carry of the bias addition (n ~ 2^256)
  static constexpr int KB_LIMBS = 9;
  static constexpr int FIX_WINDOWS = 256 / VRFS_FIX_BITS + 1;   // + the carry of the bias addition (n ~ 2^256)
  static constexpr int CARRY_WINDOWS = 1;
  static HD_INLINE void set_identity(Pt& P) { sw_set_identity(P); }
  static HD_INLINE void from_affine(Pt& P, const typename C::F& x, const typename C::F& y) { sw_from_affine<C>(P, x, y); }
  static HD_INLINE bool on_curve(const typename C::F& x, const typename C::F& y) { return sw_on_curve<C>(x, y); }
  static HD_INLINE void to_entry(Entry& e, const Pt& P) { e = P; }
  static HD_INLINE void add_entry(Pt* acc, const Entry* e, bool negate, bool = true) { Entry q = *e; sw_cneg(q, negate); sw_add<C>(acc, acc, &q); }
  static HD_INLINE void add_fix(Pt* acc, const FixEntry* e, bool negate, bool = true) { add_entry(acc, e, negate); }
  static HD_INLINE void dbl4(Pt* acc) {
    if constexpr (C::A_IS_M3) sw_dbl4_am3<C>(acc, acc);                          // secp256r1
    else { for (int i = 0; i < 4; i++) sw_add<C>(acc, acc, acc); }               // general a (bandersnatch_sw): the complete addition doubles
  }
  static HD_INLINE void dbl(Pt* acc) { sw_add<C>(acc, acc, acc); }
  static HD_INLINE void dbl_entry(Pt* r, const Entry* e) { *r = *e; sw_add<C>(r, r, r); }
  static HD_INLINE void add(Pt* r, const Pt* p, const Pt* q) { sw_add<C>(r, p, q); }
  static HD_INLINE void to_fix(FixEntry& e, const Pt& P) {            // normalise to Z = 1 (identity stays (0:1:0))
    bool inf = P.Z.is_zero();
    typename C::F zi = inv(P.Z);
    e.X = P.X * zi; e.Y = select(inf, C::F::one(), P.Y * zi); e.Z = select(inf, C::F::zero(), C::F::one());
  }
  static HD_INLINE void store_xyz(uint32_t* o, const Pt& P) { store_fp_xyz(o, P.X, P.Y, P.Z); }
  static HD_INLINE void from_xyz(Pt& P, const typename C::F& X, const typename C::F& Y, const typename C::F& Z) { P.X = X; P.Y = Y; P.Z = Z; }
  static HD_INLINE void fix_from_affine(FixEntry& e, const typename C::F& x, const typename C::F& y, bool inf) {
    e.X = select(inf, C::F::zero(), x); e.Y = select(inf, C::F::one(), y); e.Z = select(inf, C::F::zero(), C::F::one());
  }
};
#ifndef VRFS_SKIP_T
#define VRFS_SKIP_T 1                     // do not compute the T coordinate of sums nobody reads (one product per window)
#endif
#ifndef VRFS_TABLE_DOUBLINGS
#define VRFS_TABLE_DOUBLINGS 1
#endif
static constexpr int TBL_ENTRIES = 9;     // 0*P .. 8*P
static constexpr int FIX_ENTRIES = (1 << (VRFS_FIX_BITS - 1)) + 1;   // 0 .. 2^(b-1) times 2^(b w) * B
// bytes of per-thread table slab for NV variable bases
template <class C> VRFS_HD constexpr size_t slab_bytes(int nv) { return (size_t)nv * Grp<C>::SPLIT * TBL_ENTRIES * sizeof(typename Grp<C>::Entry); }
template <class C> VRFS_HD constexpr size_t fix_table_entries() { return (size_t)Grp<C>::FIX_WINDOWS * FIX_ENTRIES; }

// sc_bits: an upper bound on the scalars' bit length when the caller has one (a challenge of CHALLENGE_LEN = 16 bytes is < 2^128:
// half of the windows of c*Y and c*O are empty), 0 = full width.  Only used by the suites without GLV.
struct VarTerm { const uint8_t* pts; uint32_t pt_stride; const uint8_t* sc; uint32_t sc_stride; uint32_t negate; uint32_t sc_bits; };
struct FixTerm { const uint8_t* sc; uint32_t sc_stride; uint32_t negate; const void* table; };
struct LincombArgs {
  uint32_t n;
  VarTerm var[2];
  FixTerm fix[2];
  uint32_t* out_xyz;     // n x 3N limbs: X, Y, Z (Montgomery form)
  uint8_t* valid;        // n bytes, AND-ed with "all variable bases canonical and on the curve" (may be null)
  uint8_t* slab;         // per-thread table slabs
  uint32_t* next_item;   // device work counter (items are handed out per warp)
};

// affine x||y, 32-byte little-endian canonical each -> Montgomery; false if not canonical / not on the curve.
// Short-Weierstrass: 64 zero bytes are the identity (valid; *is_inf set).
template <class C> HD_INLINE bool load_affine(typename C::F& x, typename C::F& y, bool* is_inf, const uint8_t* p) {
  uint32_t rx[8], ry[8];
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1], c = q[2], d = q[3];
  rx[0] = a.x; rx[1] = a.y; rx[2] = a.z; rx[3] = a.w; rx[4] = b.x; rx[5] = b.y; rx[6] = b.z; rx[7] = b.w;
  ry[0] = c.x; ry[1] = c.y; ry[2] = c.z; ry[3] = c.w; ry[4] = d.x; ry[5] = d.y; ry[6] = d.z; ry[7] = d.w;
  bool ok = is_canonical<typename C::Fq>(rx) & is_canonical<typename C::Fq>(ry);
  x = to_mont<typename C::Fq>(rx); y = to_mont<typename C::Fq>(ry);
  bool inf = false;
  if (!C::IS_TE) { uint32_t o = 0; for (int i = 0; i < 8; i++) o |= rx[i] | ry[i]; inf = (o == 0); }
  if (is_inf) *is_inf = inf;
  return inf | (ok & Grp<C>::on_curve(x, y));
}
template <class C> HD_INLINE bool te_load_affine(typename C::F& x, typename C::F& y, const uint8_t* p) { return load_affine<C>(x, y, nullptr, p); }
// 32-byte little-endian scalar, reduced mod r (codec scalar_decode = from_le_bytes_mod_order) -> canonical limbs
template <class C> HD_INLINE void load_scalar_mod_r(uint32_t* k, const uint8_t* p) {
  uint32_t raw[8];
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  raw[0] = a.x; raw[1] = a.y; raw[2] = a.z; raw[3] = a.w; raw[4] = b.x; raw[5] = b.y; raw[6] = b.z; raw[7] = b.w;
  Fp<typename C::Fr> m = to_mont<typename C::Fr>(raw);
  from_mont<typename C::Fr>(k, m);
}

// table of j*B, j = 0..8; B in projective/extended coordinates.  Twisted Edwards: the even multiples are doublings of the entry
// j/2 read back from the slab (4S + 4M instead of the 9M of an addition: 2P, 4P, 6P, 8P), the odd ones add B to the point just made.
template <class C> HD_INLINE void build_table(typename Grp<C>::Entry* tbl, const typename Grp<C>::Pt& B) {
  typedef Grp<C> G;
  typename G::Pt cur; G::set_identity(cur);
  typename G::Entry cb, e;
  G::to_entry(cb, B);
  G::to_entry(e, cur); copy_words16(&tbl[0], &e);
  copy_words16(&tbl[1], &cb);
  cur = B;
#pragma unroll 1
  for (int j = 2; j <= 8; j++) {
    if (C::IS_TE && VRFS_TABLE_DOUBLINGS && (j & 1) == 0) {
      copy_words16(&e, &tbl[j >> 1]);
      G::dbl_entry(&cur, &e);
    } else {
      G::add_entry(&cur, &cb, false);
    }
    G::to_entry(e, cur); copy_words16(&tbl[j], &e);
  }
}

// acc += (-1)^neg * k * B, k = the 32-byte scalar at `sc` reduced mod r, over a signed radix-2^BITS table of B
// (fix_windows<C, BITS>() windows of (1 << (BITS - 1)) + 1 entries d * 2^(BITS w) * B).  Windows above `topw` are skipped: the caller
// knows that they hold no digit (warp-uniform).  last: nothing follows this term, so its last sum needs no T coordinate.
// FAR: the table is far larger than L1 - start every window's record on its way to L2 before the first addition.
// (lincomb_item keeps its own copy of this loop for VRFS_FIX_BITS: calling this one from there changes the code of its kernels.)
template <class C, int BITS> VRFS_HD constexpr int fix_windows() { return 256 / BITS + Grp<C>::CARRY_WINDOWS; }
template <class C, int BITS, bool FAR>
HD_INLINE void add_fixed_term(typename Grp<C>::Pt& acc, const uint8_t* sc, const void* table, bool neg, int topw, bool last) {
  typedef Grp<C> G;
  constexpr int ENTRIES = (1 << (BITS - 1)) + 1;
  uint32_t k[9];
  load_scalar_mod_r<C>(k, sc);
  k[8] = 0;
  add_window_bias<9>(k, BITS == 16 ? 0x80008000u : 0x80808080u, 8);
  const typename G::FixEntry* tbl = reinterpret_cast<const typename G::FixEntry*>(table);
  constexpr int TOPW = 256 / BITS;              // index of the carry window (short-Weierstrass suites only)
  auto digit = [&](int w) { return w == TOPW ? (int)k[8] : (BITS == 16 ? digit16(k, w) : digit8(k, w)); };
  if (FAR) {
#pragma unroll 1
    for (int w = 2; w <= topw; w++) { int dn = digit(w); prefetch_l2(&tbl[(size_t)w * ENTRIES + (dn < 0 ? -dn : dn)], sizeof(typename G::FixEntry)); }
    { int dn = digit(0); prefetch_l1(&tbl[(dn < 0 ? -dn : dn)], sizeof(typename G::FixEntry)); }
  }
#pragma unroll 1
  for (int w = 0; w <= topw; w++) {
    if (w + 1 <= topw) {              // next window's entry -> L1 while this addition runs
      int dn = digit(w + 1);
      prefetch_l1(&tbl[(size_t)(w + 1) * ENTRIES + (dn < 0 ? -dn : dn)], sizeof(typename G::FixEntry));
    }
    int d = digit(w);
    int idx = d < 0 ? -d : d;
    typename G::FixEntry e;
    copy_words16(&e, &tbl[(size_t)w * ENTRIES + idx]);
    G::add_fix(&acc, &e, (d < 0) != neg, VRFS_SKIP_T ? (!last || w != topw) : true);
  }
}

// MORE: the caller adds further terms to acc after this returns, so the last sum needs its T coordinate even when NF = 0
template <class C, int NV, int NF, bool MORE = false>
HD_INLINE bool lincomb_item(const LincombArgs& A, uint32_t item, typename Grp<C>::Entry* slab, typename Grp<C>::Pt& acc) {
  typedef Grp<C> G;
  typedef typename C::F F;
  constexpr int NT = NV * G::SPLIT;
  bool ok = true;
  G::set_identity(acc);
  if (NV > 0) {
    uint32_t kb[NT > 0 ? NT : 1][G::KB_LIMBS];
    bool kneg[NT > 0 ? NT : 1];
#pragma unroll
    for (int v = 0; v < NV; v++) {
      F x, y;
      bool inf = false;
      ok &= load_affine<C>(x, y, &inf, A.var[v].pts + (size_t)item * A.var[v].pt_stride);
      typename G::Pt B; G::from_affine(B, x, y);
      if (!C::IS_TE && inf) G::set_identity(B);
      uint32_t k[8];
      load_scalar_mod_r<C>(k, A.var[v].sc + (size_t)item * A.var[v].sc_stride);
      bool neg = A.var[v].negate != 0;
      if constexpr (C::IS_TE && G::SPLIT == 2) {
        GlvHalf h1, h2;
        band_glv_split(&h1, &h2, k);
        for (int i = 0; i < 4; i++) { kb[2 * v][i] = h1.mag[i]; kb[2 * v + 1][i] = h2.mag[i]; }
        kneg[2 * v] = h1.neg ^ neg; kneg[2 * v + 1] = h2.neg ^ neg;
        build_table<C>(slab + (2 * v) * TBL_ENTRIES, B);
        typename G::Pt E;
        G::endo(&E, &B);
        build_table<C>(slab + (2 * v + 1) * TBL_ENTRIES, E);
      } else {
        for (int i = 0; i < G::KB_LIMBS; i++) kb[v][i] = i < 8 ? k[i] : 0u;
        kneg[v] = neg;
        build_table<C>(slab + v * TBL_ENTRIES, B);
      }
    }
    for (int t = 0; t < NT; t++) add_window_bias<G::KB_LIMBS>(kb[t], 0x88888888u, G::KB_LIMBS > 8 ? 8 : G::KB_LIMBS);
    // highest window that can hold a non-zero digit, per table (+1: the bias addition may carry one window up); warp-uniform
    int topw[NT > 0 ? NT : 1], wstart = 0;
#pragma unroll
    for (int t = 0; t < NT; t++) {
      const uint32_t bits = G::SPLIT == 1 ? A.var[t].sc_bits : 0u;
      topw[t] = (bits != 0 && (int)(bits / 4 + 1) < G::WINDOWS - 1) ? (int)(bits / 4 + 1) : G::WINDOWS - 1;
      wstart = topw[t] > wstart ? topw[t] : wstart;
    }
#pragma unroll 1
    for (int w = wstart; w >= 0; w--) {
      // the table entries of this window do not depend on acc: pull them into L1 while the four doublings run
      // (the slab is L2/DRAM-resident; without this the loads below stall ~7 % of the kernel's issue slots)
#pragma unroll
      for (int t = 0; t < NT; t++) {
        int d = (G::KB_LIMBS > 8 && w == 64) ? (int)kb[t][8] : digit4(kb[t], w);
        prefetch_l1(&slab[t * TBL_ENTRIES + (d < 0 ? -d : d)], sizeof(typename G::Entry));
      }
      if (w != wstart) G::dbl4(&acc);
#pragma unroll
      for (int t = 0; t < NT; t++) {
        if (w > topw[t]) continue;
        int d = (G::KB_LIMBS > 8 && w == 64) ? (int)kb[t][8] : digit4(kb[t], w);   // the top digit is the bias carry, unbiased
        int idx = d < 0 ? -d : d;
        typename G::Entry e;
        copy_words16(&e, &slab[t * TBL_ENTRIES + idx]);
        // the last addition of a window is followed by the next window's doublings (which do not read T) or, after the last
        // window, by nothing but the fixed-base additions: its T is only computed when somebody reads it
        G::add_entry(&acc, &e, (d < 0) != kneg[t], VRFS_SKIP_T ? (t != NT - 1 || (w == 0 && (NF > 0 || MORE))) : true);
      }
    }
  }
  // fixed bases.  add_fixed_term below is the same loop with the window width and the top window as parameters (prepared keys);
  // keep the two in step - this copy stays because routing it through add_fixed_term changes the code of these kernels
#pragma unroll
  for (int f = 0; f < NF; f++) {
    uint32_t k[9];
    load_scalar_mod_r<C>(k, A.fix[f].sc + (size_t)item * A.fix[f].sc_stride);
    k[8] = 0;
    add_window_bias<9>(k, VRFS_FIX_BITS == 16 ? 0x80008000u : 0x80808080u, 8);
    const typename G::FixEntry* tbl = reinterpret_cast<const typename G::FixEntry*>(A.fix[f].table);
    bool neg = A.fix[f].negate != 0;
    constexpr int TOPW = 256 / VRFS_FIX_BITS;     // index of the carry window (short-Weierstrass suites only)
    auto digit = [&](int w) { return w == TOPW ? (int)k[8] : (VRFS_FIX_BITS == 16 ? digit16(k, w) : digit8(k, w)); };
    if (VRFS_FIX_BITS == 16) {                    // the table is far larger than L1: start every window's record on its way to L2 now
#pragma unroll 1
      for (int w = 2; w < G::FIX_WINDOWS; w++) { int dn = digit(w); prefetch_l2(&tbl[(size_t)w * FIX_ENTRIES + (dn < 0 ? -dn : dn)], sizeof(typename G::FixEntry)); }
      { int dn = digit(0); prefetch_l1(&tbl[(dn < 0 ? -dn : dn)], sizeof(typename G::FixEntry)); }
    }
#pragma unroll 1
    for (int w = 0; w < G::FIX_WINDOWS; w++) {
      if (w + 1 < G::FIX_WINDOWS) {   // next window's entry -> L1 while this addition runs
        int dn = digit(w + 1);
        prefetch_l1(&tbl[(size_t)(w + 1) * FIX_ENTRIES + (dn < 0 ? -dn : dn)], sizeof(typename G::FixEntry));
      }
      int d = digit(w);
      int idx = d < 0 ? -d : d;
      typename G::FixEntry e;
      copy_words16(&e, &tbl[(size_t)w * FIX_ENTRIES + idx]);
      G::add_fix(&acc, &e, (d < 0) != neg, VRFS_SKIP_T ? (f != NF - 1 || w != G::FIX_WINDOWS - 1) : true);
    }
  }
  return ok;
}

// ---- prepared keys: a per-key fixed-base table of 8-bit windows --------------------------------------------------------------
// U = s*G - c*Y_k of an IETF verify against a known key: two fixed-base terms and no variable base (no slab, no doublings).
static constexpr int KEY_FIX_BITS = 8;
static constexpr int KEY_ENTRIES = (1 << (KEY_FIX_BITS - 1)) + 1;   // 0 .. 128 times 256^w * Y
template <class C> VRFS_HD constexpr size_t key_table_entries() { return (size_t)fix_windows<C, KEY_FIX_BITS>() * KEY_ENTRIES; }
struct KeyedArgs {
  uint32_t n;
  const uint8_t* s;             // n x 32: s of s*G (G: the context's table of VRFS_FIX_BITS windows)
  const uint8_t* c;             // n x 32: c of -c*Y_k
  uint32_t c_bits;              // bound on c's bit length (8 * CHALLENGE_LEN), 0 = full width
  const uint32_t* key_index;    // n: k of item i (>= n_keys: the table of key 0 is read; the gather kernel rejects the item)
  uint32_t n_keys;
  const void* g_table;
  const void* key_tables;       // n_keys x key_table_entries<C>() FixEntry
  uint32_t* out_xyz;            // n x 3N limbs
};
template <class C> HD_INLINE void lincomb_keyed_item(const KeyedArgs& A, uint32_t item, typename Grp<C>::Pt& acc) {
  typedef Grp<C> G;
  uint32_t k = A.key_index[item];
  if (k >= A.n_keys) k = 0;
  const int topw_c = A.c_bits != 0 && (int)(A.c_bits / KEY_FIX_BITS) < fix_windows<C, KEY_FIX_BITS>() - 1 ? (int)(A.c_bits / KEY_FIX_BITS)
                                                                                                        : fix_windows<C, KEY_FIX_BITS>() - 1;
  G::set_identity(acc);
  add_fixed_term<C, VRFS_FIX_BITS, VRFS_FIX_BITS == 16>(acc, A.s + (size_t)item * 32, A.g_table, false, fix_windows<C, VRFS_FIX_BITS>() - 1, false);
  // n_keys x 400 KB is DRAM-resident beyond a few hundred keys: the records of all windows go to L2 up front, as for the G table
  add_fixed_term<C, KEY_FIX_BITS, true>(acc, A.c + (size_t)item * 32,
                                        reinterpret_cast<const typename G::FixEntry*>(A.key_tables) + (size_t)k * key_table_entries<C>(), true, topw_c, true);
}

// ---- prepared inputs: V = s*I_j - c*O of an IETF verify against a known VRF input ---------------------------------------------
// I_j has a table of the prepared-key layout (vrfs_inputs_prepare), so s*I_j is 32-33 mixed additions; c*O stays the variable-base
// Straus loop of lincomb_item<C, 1, 0> (GLV halves on Bandersnatch, sc_bits-trimmed windows for a 16-byte challenge) on a slab of
// one base.  L.var[0] = the c*O term, L.fix[0] = the s*I term with `table` = the n_inputs tables back to back.
struct IoArgs {
  LincombArgs L;
  const uint32_t* input_index;  // n: j of item i (>= n_inputs: the table of input 0 is read; the gather kernel rejects the item)
  uint32_t n_inputs;
};
template <class C>
HD_INLINE bool lincomb_io_item(const IoArgs& A, uint32_t item, typename Grp<C>::Entry* slab, typename Grp<C>::Pt& acc) {
  typedef Grp<C> G;
  const bool ok = lincomb_item<C, 1, 0, true>(A.L, item, slab, acc);
  uint32_t j = A.input_index[item];
  if (j >= A.n_inputs) j = 0;
  const FixTerm& f = A.L.fix[0];
  // FAR: up to 65536 tables of ~400 KB, far larger than L2 - as for the key tables of lincomb_keyed_item
  add_fixed_term<C, KEY_FIX_BITS, true>(acc, f.sc + (size_t)item * f.sc_stride,
                                        reinterpret_cast<const typename G::FixEntry*>(f.table) + (size_t)j * key_table_entries<C>(), f.negate != 0,
                                        fix_windows<C, KEY_FIX_BITS>() - 1, true);
  return ok;
}

// one fixed-base table entry: (d * 256^w) * B.  Used once per context by the table kernel.
template <class C>
HD_INLINE void fixed_table_entry(typename Grp<C>::FixEntry& out, const typename C::F& bx, const typename C::F& by, int w, int d) {
  typedef Grp<C> G;
  typename G::Pt P, R; G::from_affine(P, bx, by);
  for (int i = 0; i < VRFS_FIX_BITS * w; i++) G::dbl(&P);
  G::set_identity(R);
  for (int bit = VRFS_FIX_BITS - 1; bit >= 0; bit--) {
    G::dbl(&R);
    if ((d >> bit) & 1) G::add(&R, &R, &P);
  }
  G::to_fix(out, R);
}

// Prepared-key tables, layout [key][window][entry]: entry d of window w is d * 256^w * Y.  k_fixed_table's scheme (a doubling
// chain of its own per entry) is fine for two bases and far too slow for millions of entries; instead
//  1. key_table_powers: one doubling chain per key gives 256^w * Y for every w, parked as (X : Y : Z) in entry 1 of window w;
//  2. key_table_window: one thread per window makes d * 256^w * Y, d = 2..128, by successive additions and normalises all of
//     them with ONE inversion.  Montgomery's trick without a prefix array: the forward pass stores (X_d P_(d-1), Y_d P_(d-1), Z_d)
//     with P_d = Z_1 ... Z_d, so that x_d = X_d P_(d-1) / P_d; the backward pass walks 1 / P_d down from 1 / P_128 with Z_d.
// A key that is not valid gets the identity's table.  Returns whether the key is valid (key_ok).
template <class C> HD_INLINE bool key_table_powers(typename Grp<C>::FixEntry* tbl, const uint8_t* pk) {
  typedef Grp<C> G;
  typedef typename C::F F;
  F x, y;
  bool inf = false;
  const bool ok = load_affine<C>(x, y, &inf, pk) && !inf;   // the short-Weierstrass identity is a valid point but no key
  typename G::Pt P;
  if (ok) G::from_affine(P, x, y); else G::set_identity(P);
#pragma unroll 1
  for (int w = 0; w < fix_windows<C, KEY_FIX_BITS>(); w++) {
    F* slot = reinterpret_cast<F*>(&tbl[(size_t)w * KEY_ENTRIES + 1]);
    slot[0] = P.X; slot[1] = P.Y; slot[2] = P.Z;
    if (w + 1 < fix_windows<C, KEY_FIX_BITS>()) { G::dbl4(&P); G::dbl4(&P); }
  }
  return ok;
}
template <class C> HD_INLINE void key_table_window(typename Grp<C>::FixEntry* win) {
  typedef Grp<C> G;
  typedef typename C::F F;
  F* s1 = reinterpret_cast<F*>(&win[1]);
  typename G::Pt B, cur;
  G::from_xyz(B, s1[0], s1[1], s1[2]);
  typename G::Entry eb;
  G::to_entry(eb, B);
  cur = B;
  F pre = F::one();
#pragma unroll 1
  for (int d = 1; d < KEY_ENTRIES; d++) {
    if (d > 1) G::add_entry(&cur, &eb, false);
    F* slot = reinterpret_cast<F*>(&win[d]);
    slot[0] = cur.X * pre; slot[1] = cur.Y * pre; slot[2] = cur.Z;
    pre = pre * select(cur.Z.is_zero(), F::one(), cur.Z);     // the short-Weierstrass identity (Z = 0) stays out of the chain
  }
  F acc = inv(pre);
#pragma unroll 1
  for (int d = KEY_ENTRIES - 1; d >= 1; d--) {
    F* slot = reinterpret_cast<F*>(&win[d]);
    const F X = slot[0], Y = slot[1], Z = slot[2];
    const bool zero = Z.is_zero();
    typename G::FixEntry e;
    G::fix_from_affine(e, X * acc, Y * acc, zero);
    acc = acc * select(zero, F::one(), Z);
    win[d] = e;
  }
  typename G::FixEntry e0;
  G::fix_from_affine(e0, F::zero(), F::one(), true);
  win[0] = e0;
}

}  // namespace vrfs
