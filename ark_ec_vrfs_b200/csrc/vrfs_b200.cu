// vrfs_b200: kernels + the C ABI of include/vrfs_b200.h.  sm_100a only; no CPU fallback - every entry
// point launches kernels on the context's device and reports CUDA failures as VRFS_CUDA_ERROR.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdint.h>
#include <stdlib.h>
#include <algorithm>
#include <memory>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/vrfs_b200.h"
#include "h2c.cuh"
#include "wire.cuh"
#include "msm.cuh"
#include "te_msm.cuh"
#include "ring.cuh"
#include "g1_fft.cuh"
#include "pairing_coop.cuh"

using namespace vrfs;

// =================================================================================================
// kernels
// =================================================================================================
// launch shape of the lincomb kernels: measured on B200 (tools/cfg_probe.sh) 256x2 > 128x5 > 128x4 > 128x3, all within 4 %
#ifndef LINCOMB_THREADS
#define LINCOMB_THREADS 256
#endif
#ifndef LINCOMB_MINBLOCKS
#define LINCOMB_MINBLOCKS 2
#endif
#ifndef VRFS_MSM_TAIL_16THS
#define VRFS_MSM_TAIL_16THS 2            // sixteenths of the buckets of a large STATELESS MSM accumulated by the short-task tail launch (0 = off)
#endif
#ifndef VRFS_PAIR_WAVES
#define VRFS_PAIR_WAVES 6                // verify batches below this many resident waves run both linear combinations in one grid (0 = never)
#endif
#ifndef VRFS_SPLIT_ITEMS_PER_SM
#define VRFS_SPLIT_ITEMS_PER_SM 256      // a verify batch of up to this many items per SM runs its two linear combinations on two streams
#endif

// one fixed-base table (K8): thread (w, d) computes (d * 256^w) * B in affine cached form
template <class C>
__global__ void k_fixed_table(typename Grp<C>::FixEntry* out, int blinding) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int)fix_table_entries<C>()) return;
  int w = t / FIX_ENTRIES, d = t % FIX_ENTRIES;
  typename Grp<C>::FixEntry e;
  fixed_table_entry<C>(e, blinding ? C::bx() : C::gx(), blinding ? C::by() : C::gy(), w, d);
  out[t] = e;
}

// K7/K8/K9a: R_i = sum var + sum fixed, projective out.  Persistent grid-stride so that the window-table
// slab is per resident thread (L2-resident), not per item.
template <class C, int NV, int NF>
__global__ void __launch_bounds__(LINCOMB_THREADS, LINCOMB_MINBLOCKS) k_lincomb(LincombArgs A) {
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31u;
  typename Grp<C>::Entry* slab = reinterpret_cast<typename Grp<C>::Entry*>(A.slab + (size_t)tid * slab_bytes<C>(NV));
  // items are handed out 32 at a time per warp from a device counter: no tail wave of idle warps behind the slowest SMs
  for (;;) {
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(A.next_item, 32u);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base >= A.n) break;
    const uint32_t item = base + lane;
    if (item < A.n) {
      typename Grp<C>::Pt acc;
      bool ok = lincomb_item<C, NV, NF>(A, item, slab, acc);
      Grp<C>::store_xyz(A.out_xyz + (size_t)item * 24, acc);
      if (A.valid != nullptr && !ok) A.valid[item] = 0;
    }
    __syncwarp();
  }
}

// Both linear combinations of a verify batch in ONE grid: U = s*G - c*Y (<1,1>) and V = s*I - c*O (<2,0>) as 2 * ceil(n/32) warp
// tasks handed out from one counter, the long ones (V) first.  A mid-size batch - what one GPU gets when a caller spreads 2^20 items
// over eight - is 1.7 resident waves of each kernel: two launches round that up to 2 + 2 half-empty waves, one task queue does not.
template <class C>
__global__ void __launch_bounds__(LINCOMB_THREADS, LINCOMB_MINBLOCKS) k_lincomb_verify_pair(LincombArgs U, LincombArgs V) {
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31u;
  typename Grp<C>::Entry* slab = reinterpret_cast<typename Grp<C>::Entry*>(V.slab + (size_t)tid * slab_bytes<C>(2));
  const uint32_t groups = (V.n + 31u) / 32u;
  for (;;) {
    uint32_t task = 0;
    if (lane == 0) task = atomicAdd(V.next_item, 1u);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= 2u * groups) break;
    const bool is_v = task < groups;                      // warp-uniform
    const uint32_t item = (is_v ? task : task - groups) * 32u + lane;
    if (item < V.n) {
      typename Grp<C>::Pt acc;
      if (is_v) {
        const bool ok = lincomb_item<C, 2, 0>(V, item, slab, acc);
        Grp<C>::store_xyz(V.out_xyz + (size_t)item * 24, acc);
        if (V.valid != nullptr && !ok) V.valid[item] = 0;
      } else {
        const bool ok = lincomb_item<C, 1, 1>(U, item, slab, acc);
        Grp<C>::store_xyz(U.out_xyz + (size_t)item * 24, acc);
        if (U.valid != nullptr && !ok) U.valid[item] = 0;
      }
    }
    __syncwarp();
  }
}

// K9b: inversion shared by FINISH_K items per thread (Montgomery's trick), 5 point encodings, challenge hash, compare
#define FINISH_K 8
template <class S>
__global__ void __launch_bounds__(128) k_ietf_verify_finish(uint32_t n, const uint8_t* pk, const uint8_t* input, const uint8_t* output,
                                                             const uint8_t* c, const uint32_t* u_xyz, const uint32_t* v_xyz,
                                                             const uint8_t* ad, const uint64_t* ad_off, const uint8_t* valid, uint8_t* out_ok, uint8_t* out_status) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  if (t >= n) return;
  ietf_verify_finish_batched<S, FINISH_K>(n, t, stride, pk, input, output, c, u_xyz, v_xyz, ad, ad_off, valid, out_ok, out_status);
}

// prepared public keys (vrfs_public_keys_prepare): the per-key 8-bit tables (lincomb.cuh "Prepared-key tables"), the keyed U = s*G - c*Y_k,
// and the gather of each item's key row for k_ietf_verify_finish
template <class C>
__global__ void __launch_bounds__(128) k_key_table_powers(uint32_t n_keys, const uint8_t* pks, typename Grp<C>::FixEntry* tables, uint8_t* rows, uint8_t* key_ok) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_keys) return;
  key_ok[k] = key_table_powers<C>(tables + (size_t)k * key_table_entries<C>(), pks + (size_t)64 * k);
  copy_words16(reinterpret_cast<uint4(*)[4]>(rows) + k, reinterpret_cast<const uint4(*)[4]>(pks) + k);
}
template <class C>
__global__ void __launch_bounds__(128) k_key_table_windows(uint32_t n_keys, typename Grp<C>::FixEntry* tables) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_keys * (uint32_t)fix_windows<C, KEY_FIX_BITS>()) return;
  key_table_window<C>(tables + (size_t)t * KEY_ENTRIES);      // windows of consecutive keys are contiguous
}
// 128-thread blocks: the short-Weierstrass suites need ~134 registers to run without spills (3 blocks, 12 warps per SM); the
// twisted-Edwards ones fit 128 registers and keep the 16 warps per SM of k_lincomb
#define KEYED_THREADS 128
template <class C>
__global__ void __launch_bounds__(KEYED_THREADS, C::IS_TE ? 4 : 3) k_lincomb_keyed(KeyedArgs A) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;   // every item costs the same: a plain grid, no work counter
  if (i >= A.n) return;
  typename Grp<C>::Pt acc;
  lincomb_keyed_item<C>(A, i, acc);
  Grp<C>::store_xyz(A.out_xyz + (size_t)i * 24, acc);
}
// item i's key row (zeros for an index out of range); valid[i] = 0 for such an index or a key that is not valid
__global__ void __launch_bounds__(128) k_gather_keys(uint32_t n, const uint32_t* key_index, uint32_t n_keys, const uint8_t* rows, const uint8_t* key_ok,
                                                     uint8_t* out_rows, uint8_t* valid) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t k = key_index[i];
  uint4 r[4] = {};
  if (k < n_keys) copy_words16(&r, reinterpret_cast<const uint4(*)[4]>(rows) + k);
  copy_words16(reinterpret_cast<uint4(*)[4]>(out_rows) + i, &r);
  if (k >= n_keys || !key_ok[k]) valid[i] = 0;
}
// prepared inputs (vrfs_inputs_prepare): V = s*I_j - c*O (lincomb.cuh lincomb_io_item) on the persistent grid of k_lincomb - the
// variable base c*O needs a window-table slab, which the grid keeps per resident thread instead of per item.  128-thread blocks:
// at 128 registers the variable-base loop spills on Bandersnatch (GLV) and the short-Weierstrass suites, as k_lincomb<C, 1, 0>
// does; 3 blocks per SM (12 warps) give them ~170 registers and no spills, the other twisted-Edwards suites keep 16 warps.
#define IO_THREADS 128
template <class C> constexpr int io_min_blocks() { return C::IS_TE && Grp<C>::SPLIT == 1 ? 4 : 3; }
template <class C>
__global__ void __launch_bounds__(IO_THREADS, io_min_blocks<C>()) k_lincomb_io(IoArgs A) {
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31u;
  typename Grp<C>::Entry* slab = reinterpret_cast<typename Grp<C>::Entry*>(A.L.slab + (size_t)tid * slab_bytes<C>(1));
  for (;;) {
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(A.L.next_item, 32u);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base >= A.L.n) break;
    const uint32_t item = base + lane;
    if (item < A.L.n) {
      typename Grp<C>::Pt acc;
      const bool ok = lincomb_io_item<C>(A, item, slab, acc);
      Grp<C>::store_xyz(A.L.out_xyz + (size_t)item * 24, acc);
      if (A.L.valid != nullptr && !ok) A.L.valid[item] = 0;
    }
    __syncwarp();
  }
}

// integer-pipe roofline microbenchmarks (SURVEY 8d): independent multiply-accumulate chains per thread
template <int VARIANT>
__global__ void __launch_bounds__(256) k_mac_bench(uint32_t* out, int iters, unsigned long long* cycles) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long c0 = clock64();
  // NOTE: every multiply below takes one operand from its own accumulator.  With loop-invariant multiplicands ptxas
  // hoists the product and the loop measures 64-bit ADDs (that mistake gave a bogus 18.5 T "peak" in profiles/r1a_*).
  if (VARIANT == 0) {          // IMAD.WIDE.U32: acc = lo(acc) * y + acc, 8 independent chains
    unsigned long long a[8];
    for (int k = 0; k < 8; k++) a[k] = ((unsigned long long)(t * 2654435761u + k) << 32) | (t + k * 40503u + 1u);
    uint32_t y = (t ^ 0x9e3779b9u) | 1u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int r = 0; r < 4; r++)
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = (unsigned long long)(uint32_t)a[k] * y + a[k];
    }
    unsigned long long s = 0;
    for (int k = 0; k < 8; k++) s ^= a[k];
    out[t] = (uint32_t)s ^ (uint32_t)(s >> 32);
  } else if (VARIANT == 1) {   // IMAD (32-bit): acc = acc * y + x
    uint32_t a[8];
    for (int k = 0; k < 8; k++) a[k] = t * 2654435761u + k * 40503u + 1u;
    uint32_t y = (t ^ 0x9e3779b9u) | 1u, x = t + 12345u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int r = 0; r < 4; r++)
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = a[k] * y + x;
    }
    uint32_t s = 0;
    for (int k = 0; k < 8; k++) s ^= a[k];
    out[t] = s;
  } else if (VARIANT == 2) {   // dependent chain of BLS12-381 Fr Montgomery products (136 MAC32 each); 32 per iteration
    Fp<BlsFr> a, b;
    for (int i = 0; i < 8; i++) { a.v[i] = t + i; b.v[i] = (t ^ 0x5bd1e995u) + 7 * i; }
    a.v[7] &= 0x3fffffffu; b.v[7] &= 0x3fffffffu;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll 1
      for (int r = 0; r < 16; r++) { a = a * b; b = b * a; }
    }
    uint32_t s = 0;
    for (int i = 0; i < 8; i++) s ^= a.v[i] ^ b.v[i];
    out[t] = s;
  } else if (VARIANT == 3) {   // two independent chains of products per thread (more ILP)
    Fp<BlsFr> a, b, c, d;
    for (int i = 0; i < 8; i++) { a.v[i] = t + i; b.v[i] = (t ^ 0x5bd1e995u) + 7 * i; c.v[i] = t * 3 + i; d.v[i] = t * 5 + i; }
    a.v[7] &= 0x3fffffffu; b.v[7] &= 0x3fffffffu; c.v[7] &= 0x3fffffffu; d.v[7] &= 0x3fffffffu;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll 1
      for (int r = 0; r < 8; r++) { a = a * b; c = c * d; b = b * a; d = d * c; }
    }
    uint32_t s = 0;
    for (int i = 0; i < 8; i++) s ^= a.v[i] ^ b.v[i] ^ c.v[i] ^ d.v[i];
    out[t] = s;
  } else if (VARIANT == 5 || VARIANT == 6) {   // 4 independent 8-limb carry chains (the multiplier's row shape); 6: immediate multiplicand
    uint32_t acc[4][8], top[4], x[8];
    for (int c = 0; c < 4; c++) { top[c] = 0; for (int i = 0; i < 8; i++) acc[c][i] = t * (c + 3) + i; }
    for (int i = 0; i < 8; i++) x[i] = VARIANT == 5 ? (t ^ (0x9e3779b9u * (i + 1))) : BlsFr::mod(i);
    uint32_t y = t * 2654435761u + 12345u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int r = 0; r < 2; r++) {
#pragma unroll
        for (int c = 0; c < 4; c++) MontChains<8>::mad_row(acc[c], top[c], x, y + c);
      }
    }
    uint32_t s = 0;
    for (int c = 0; c < 4; c++) { s ^= top[c]; for (int i = 0; i < 8; i++) s ^= acc[c][i]; }
    out[t] = s;
  } else if (VARIANT == 9) {   // DFMA: acc = fma(acc, y, x) with round-toward-zero, 8 independent chains (FP64 pipe)
    double a[8];
    for (int k = 0; k < 8; k++) a[k] = 1.0 + (double)((t + k) & 1023) * 1e-3;
    double y = __longlong_as_double(0x3ff0000000000000ll | (long long)(t & 0xffff)), x = (double)(t & 7) * 1e-9;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int r = 0; r < 4; r++)
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = __fma_rz(a[k], y, x);
    }
    double s = 0;
    for (int k = 0; k < 8; k++) s += a[k];
    out[t] = (uint32_t)__double2loint(s) ^ (uint32_t)__double2hiint(s);
  } else {                     // VARIANT 4: IMAD.HI.U32: acc = hi(acc * y) + x
    uint32_t a[8];
    for (int k = 0; k < 8; k++) a[k] = t * 2654435761u + k * 40503u + 0x80000001u;
    uint32_t y = (t ^ 0x9e3779b9u) | 0xc0000000u, x = t + 12345u;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
      for (int r = 0; r < 4; r++)
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = __umulhi(a[k], y) + x;
    }
    uint32_t s = 0;
    for (int k = 0; k < 8; k++) s ^= a[k];
    out[t] = s;
  }
  unsigned long long c1 = clock64();
  if (threadIdx.x == 0 && blockIdx.x == 0) *cycles = c1 - c0;
}

// =================================================================================================
// context
// =================================================================================================
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  size_t secret_bytes = 0;   // > 0: the running call put key material here (sk, nonces, blinding factors); zeroed before it returns
};
enum { BUF_IN0, BUF_IN1, BUF_IN2, BUF_IN3, BUF_IN4, BUF_AD, BUF_OFF, BUF_OUT0, BUF_OUT1, BUF_W0, BUF_W1, BUF_W2, BUF_W3, BUF_VALID, BUF_SLAB,
       BUF_X0, BUF_X1, BUF_X2, BUF_X3, BUF_X4, BUF_X5, BUF_ZINV, BUF_SLAB2,
       BUF_PB0, BUF_PB1, BUF_PB2, BUF_KEYROWS, BUF_INROWS, BUF_COUNT };   // X*: wire-format staging (encoded keys, signatures, h2c data, flags); PB*: Pedersen batch verification;
                                                             // KEYROWS / INROWS: the key / input rows a prepared verify gathers for its finish kernel

#define MAX_TIMED 64
#ifndef VRFS_HOST_PIECES
#define VRFS_HOST_PIECES 6   // host-buffer calls: at most this many pieces per batch (stage_in_pieces)
#endif
struct vrfs_ctx {
  int device = 0, sms = 0;
  bool timing = false;
  int n_timed = 0;
  cudaEvent_t tev[MAX_TIMED + 1] = {nullptr};
  const char* tname[MAX_TIMED] = {nullptr};
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;                 // H2D of later chunks overlaps the kernels of earlier ones
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;   // kernels on copy_stream beside the main stream (side_fork / side_join)
  cudaEvent_t ev_in[VRFS_HOST_PIECES] = {nullptr}, ev_out[VRFS_HOST_PIECES] = {nullptr};   // per-piece host transfers (stage_in_pieces / pieces_copy_out)
  char err[512] = {0};
  std::recursive_mutex mu;            // entry points serialise per context (SURVEY 8b: "internally synchronised")
  uint64_t launches = 0;
  int depth = 0;                      // nesting of entry points on this context (a host-buffer call runs its *_dev form inside)
  bool failed = false;                // the running call hit an error: both streams are drained before it returns
  DevBuf buf[BUF_COUNT];
  void* fixtab[VRFS_SUITE_COUNT][2] = {};   // [suite][G | blinding base], built on first use
  std::vector<struct vrfs_msm_bases*> prepared;   // live prepared-base handles (freed / orphaned by vrfs_ctx_destroy)
  std::vector<struct vrfs_public_keys*> prepared_keys;   // live prepared-key handles (likewise)
  // peer group of the multi-GPU MSM exchange (csrc/msm.cuh "multi-GPU exchange"): world = 0 until connected
  struct {
    int rank = 0, world = 0;
    unsigned long long epoch = 0;
    PeerBox* box[VRFS_MAX_PEERS] = {nullptr};      // box[rank] = this GPU's own mailbox (cudaMalloc); the others mapped
    bool ipc[VRFS_MAX_PEERS] = {false};            // mapped through cudaIpcOpenMemHandle (to be closed), not a same-process pointer
    unsigned int* timed_out = nullptr;             // mapped pinned host word written by a kernel that gave up waiting
    unsigned long long timeout_ns = 2000000000ull;
  } peer;
};

static vrfs_status fail(vrfs_ctx* c, vrfs_status st, const char* fmt, ...) {
  if (c) { va_list ap; va_start(ap, fmt); vsnprintf(c->err, sizeof c->err, fmt, ap); va_end(ap); c->failed = true; }
  return st;
}
// Every entry point holds one of these: the per-context lock plus the end-of-call hygiene of the OUTERMOST call -
//  * device buffers that held key material (DevBuf::secret_bytes) are zeroed and the stream drained (SURVEY 8b: "staging buffers
//    holding sk are zeroed before release"; the buffers are pooled, so "release" is the end of the call);
//  * after a failure both streams are drained, so that no copy is still reading the caller's host buffers when the error
//    code reaches the caller.
// An entry point passes its name (__func__): one NVTX range per ABI call, named after the entry point (`ncu --nvtx --nvtx-include
// "vrfs_ietf_verify_batch/"` profiles the kernels of one kind of call; header-only NVTX 3: a no-op unless a tool is attached).
struct CallGuard {
  vrfs_ctx* ctx;
  const char* range;
  explicit CallGuard(vrfs_ctx* c, const char* name = nullptr) : ctx(c), range(name) {
    ctx->mu.lock(); if (ctx->depth++ == 0) ctx->failed = false; if (range) nvtxRangePushA(range); }
  ~CallGuard() {
    if (range) nvtxRangePop();
    if (--ctx->depth == 0) {
      bool wiped = false;
      for (int i = 0; i < BUF_COUNT; i++) {
        DevBuf& b = ctx->buf[i];
        if (b.secret_bytes && b.p) { cudaMemsetAsync(b.p, 0, b.secret_bytes < b.cap ? b.secret_bytes : b.cap, ctx->stream); wiped = true; }
        b.secret_bytes = 0;
      }
      if (ctx->failed && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
      if ((wiped || ctx->failed) && ctx->stream) cudaStreamSynchronize(ctx->stream);
    }
    ctx->mu.unlock();
  }
};
#define CU(call)                                                                                                   \
  do {                                                                                                             \
    cudaError_t e_ = (call);                                                                                       \
    if (e_ != cudaSuccess) return fail(ctx, VRFS_CUDA_ERROR, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)
#define ST(call)                          \
  do {                                    \
    vrfs_status s_ = (call);              \
    if (s_ != VRFS_OK) return s_;         \
  } while (0)
// bookkeeping after every kernel launch: count it, surface launch errors, and (when kernel timing is on)
// drop an event so that bench.py can read each kernel's device time from the stream it ran on
#define LAUNCHED(ctx) do { (ctx)->launches++; CU(cudaGetLastError()); ST(note_kernel((ctx), __func__)); } while (0)
#define LAUNCHED_AS(ctx, name) do { (ctx)->launches++; CU(cudaGetLastError()); ST(note_kernel((ctx), (name))); } while (0)
static vrfs_status note_kernel(vrfs_ctx* ctx, const char* name);
static vrfs_status timing_begin(vrfs_ctx* ctx);
static void orphan_prepared(vrfs_ctx* ctx);
static void orphan_public_keys(vrfs_ctx* ctx);
static void peer_teardown(vrfs_ctx* ctx);

static vrfs_status timing_begin(vrfs_ctx* ctx) {
  ctx->n_timed = 0;
  if (!ctx->timing) return VRFS_OK;
  if (!ctx->tev[0]) for (int i = 0; i <= MAX_TIMED; i++) CU(cudaEventCreate(&ctx->tev[i]));
  CU(cudaEventRecord(ctx->tev[0], ctx->stream));
  return VRFS_OK;
}
static vrfs_status note_kernel(vrfs_ctx* ctx, const char* name) {
  if (!ctx->timing || !ctx->tev[0] || ctx->n_timed >= MAX_TIMED) return VRFS_OK;
  ctx->tname[ctx->n_timed] = name;
  ctx->n_timed++;
  CU(cudaEventRecord(ctx->tev[ctx->n_timed], ctx->stream));
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ctx_enable_kernel_timing(vrfs_ctx* ctx, int on) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ctx->timing = on != 0;
  ctx->n_timed = 0;
  return VRFS_OK;
}
// device time of every kernel of the most recent *_batch / *_batch_dev call (after a sync); returns the count
extern "C" int vrfs_ctx_kernel_timings(vrfs_ctx* ctx, const char** names, float* ms, int cap) {
  if (!ctx || !ctx->timing) return 0;
  CallGuard guard_(ctx, __func__);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return 0;
  int n = ctx->n_timed < cap ? ctx->n_timed : cap;
  for (int i = 0; i < n; i++) {
    names[i] = ctx->tname[i];
    if (cudaEventElapsedTime(&ms[i], ctx->tev[i], ctx->tev[i + 1]) != cudaSuccess) ms[i] = -1.f;
  }
  return n;
}

static vrfs_status ensure(vrfs_ctx* ctx, int which, size_t bytes, void** out) {
  DevBuf& b = ctx->buf[which];
  if (bytes == 0) bytes = 16;
  if (b.cap < bytes) {
    if (b.p) {
      if (b.secret_bytes) CU(cudaMemsetAsync(b.p, 0, b.secret_bytes < b.cap ? b.secret_bytes : b.cap, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream)); CU(cudaFree(b.p)); b.p = nullptr; b.cap = 0;
    }
    size_t cap = bytes + bytes / 8 + 256;
    CU(cudaMalloc(&b.p, cap));
    b.cap = cap;
  }
  *out = b.p;
  return VRFS_OK;
}
static inline bool aligned16(const void* p) { return (((uintptr_t)p) & 15u) == 0; }

// Fixed-base tables (G and the Pedersen blinding base B) are built the first time a suite needs them: 2 x 50 MB and ~30 ms of
// k_fixed_table per suite that a caller of one suite should not pay three times at context creation.
template <class S>
static vrfs_status need_tables(vrfs_ctx* ctx) {
  typedef typename S::C C;
  if (ctx->fixtab[S::ID][1]) return VRFS_OK;
  const int n = (int)fix_table_entries<C>();
  for (int b = 0; b < 2; b++) {
    if (ctx->fixtab[S::ID][b]) continue;
    void* t = nullptr;
    CU(cudaMalloc(&t, sizeof(typename Grp<C>::FixEntry) * n));
    k_fixed_table<C><<<(n + 63) / 64, 64, 0, ctx->stream>>>(reinterpret_cast<typename Grp<C>::FixEntry*>(t), b);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(t); return fail(ctx, VRFS_CUDA_ERROR, "k_fixed_table launch failed: %s", cudaGetErrorString(e)); }
    ST(note_kernel(ctx, "fixed_table"));
    ctx->fixtab[S::ID][b] = t;
  }
  return VRFS_OK;
}

static_assert((int)ITEM_OK == (int)VRFS_ITEM_OK && (int)ITEM_VERIFICATION_FAILURE == (int)VRFS_ITEM_VERIFICATION_FAILURE &&
              (int)ITEM_INVALID_DATA == (int)VRFS_ITEM_INVALID_DATA, "device-side status codes must match include/vrfs_b200.h");
extern "C" int vrfs_abi_version(void) { return 2; }

extern "C" vrfs_status vrfs_ctx_create(int device, vrfs_ctx** out) {
  if (!out) return VRFS_BAD_ARG;
  *out = nullptr;
  vrfs_ctx* ctx = new (std::nothrow) vrfs_ctx();
  if (!ctx) return VRFS_CUDA_ERROR;
  *out = ctx;   // returned even on failure so that vrfs_last_error can be read; destroy it either way
  ctx->device = device;
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(ctx, VRFS_CUDA_ERROR, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  ctx->sms = prop.multiProcessorCount;
  CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  for (int i = 0; i < VRFS_HOST_PIECES; i++) { CU(cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&ctx->ev_out[i], cudaEventDisableTiming)); }
  CU(cudaEventCreate(&ctx->ev0));
  CU(cudaEventCreate(&ctx->ev1));
  return VRFS_OK;                      // fixed-base tables: built on first use per suite (need_tables)
}
extern "C" void vrfs_ctx_destroy(vrfs_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  orphan_prepared(ctx);
  orphan_public_keys(ctx);
  peer_teardown(ctx);
  for (int i = 0; i < BUF_COUNT; i++) if (ctx->buf[i].p) cudaFree(ctx->buf[i].p);
  for (int s = 0; s < VRFS_SUITE_COUNT; s++) for (int b = 0; b < 2; b++) if (ctx->fixtab[s][b]) cudaFree(ctx->fixtab[s][b]);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  for (int i = 0; i < VRFS_HOST_PIECES; i++) { if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]); if (ctx->ev_out[i]) cudaEventDestroy(ctx->ev_out[i]); }
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}
extern "C" vrfs_status vrfs_ctx_sync(vrfs_ctx* ctx) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  CU(cudaStreamSynchronize(ctx->stream));
  return VRFS_OK;
}
// Page-locked host memory for callers that have no CUDA runtime of their own (a Rust shim): the batch calls copy straight from / into
// the caller's buffers, and only page-locked ones let those copies run beside the kernels.  No context involved (portable across devices).
extern "C" vrfs_status vrfs_host_alloc(size_t bytes, void** out) {
  if (!out) return VRFS_BAD_ARG;
  *out = nullptr;
  if (bytes == 0) return VRFS_OK;
  return cudaHostAlloc(out, bytes, cudaHostAllocPortable) == cudaSuccess ? VRFS_OK : (cudaGetLastError(), VRFS_CUDA_ERROR);
}
extern "C" vrfs_status vrfs_host_free(void* p) {
  if (!p) return VRFS_OK;
  return cudaFreeHost(p) == cudaSuccess ? VRFS_OK : (cudaGetLastError(), VRFS_BAD_ARG);
}
extern "C" vrfs_status vrfs_host_register(void* p, size_t bytes) {
  if (!p || bytes == 0) return VRFS_BAD_ARG;
  return cudaHostRegister(p, bytes, cudaHostRegisterPortable) == cudaSuccess ? VRFS_OK : (cudaGetLastError(), VRFS_CUDA_ERROR);
}
extern "C" vrfs_status vrfs_host_unregister(void* p) {
  if (!p) return VRFS_BAD_ARG;
  return cudaHostUnregister(p) == cudaSuccess ? VRFS_OK : (cudaGetLastError(), VRFS_BAD_ARG);
}
// test hook: bytes of an internal staging buffer (slot = position in the buffer pool; 0..4 are the input staging buffers in call
// order, e.g. slot 0 holds `sk` during a prove call).  tests/ use it to check that key material is gone after a call returned.
extern "C" vrfs_status vrfs_ctx_debug_read_staging(vrfs_ctx* ctx, int slot, size_t offset, uint8_t* out, size_t n) {
  if (!ctx || !out) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (slot < 0 || slot >= BUF_COUNT) return fail(ctx, VRFS_BAD_ARG, "no such staging buffer");
  const DevBuf& b = ctx->buf[slot];
  if (!b.p || offset + n > b.cap) return fail(ctx, VRFS_BAD_ARG, "range outside the staging buffer (capacity %zu)", b.cap);
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaMemcpy(out, (const uint8_t*)b.p + offset, n, cudaMemcpyDeviceToHost));
  return VRFS_OK;
}
extern "C" const char* vrfs_last_error(const vrfs_ctx* ctx) { return ctx ? ctx->err : "null context"; }
extern "C" void* vrfs_ctx_stream(vrfs_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" uint64_t vrfs_ctx_launch_count(const vrfs_ctx* ctx) { return ctx ? ctx->launches : 0; }
// the suite behind a vrfs_suite value, handed to a generic lambda as a value of its tag type; `unknown()` for any other value
template <class F, class U> static auto suite_switch(vrfs_suite s, F&& f, U&& unknown) -> decltype(unknown()) {
  switch (s) {
    case VRFS_BANDERSNATCH_ELL2: return f(BandSuite{});
    case VRFS_ED25519_TAI: return f(EdSuite{});
    case VRFS_P256_TAI: return f(P256Suite{});
    case VRFS_BANDERSNATCH_SW_TAI: return f(BandSwSuite{});
    case VRFS_JUBJUB_TAI: return f(JubSuite{});
    case VRFS_BABYJUBJUB_TAI: return f(BjjSuite{});
    default: return unknown();
  }
}
template <class F> static vrfs_status with_suite(vrfs_ctx* ctx, vrfs_suite s, F&& f) {
  return suite_switch(s, f, [&] { return fail(ctx, VRFS_BAD_ARG, "unknown suite %d", (int)s); });
}
template <class F> static int suite_const(vrfs_suite s, F&& f) { return suite_switch(s, f, [] { return 0; }); }
// after the argument checks of a batch entry point, before anything is enqueued
static vrfs_status begin_call(vrfs_ctx* ctx, size_t n) {
  if (n > 0x7fffffffu) return fail(ctx, VRFS_BAD_ARG, "batch too large (n < 2^31)");
  CU(cudaSetDevice(ctx->device));
  return timing_begin(ctx);
}
// ... of one that takes a suite: an unknown suite is VRFS_BAD_ARG here, before any size is derived from it
static vrfs_status begin_call(vrfs_ctx* ctx, vrfs_suite suite, size_t n) {
  ST(with_suite(ctx, suite, [](auto) { return VRFS_OK; }));
  return begin_call(ctx, n);
}
extern "C" int vrfs_suite_challenge_len(vrfs_suite s) { return suite_const(s, [](auto S_) { return (int)decltype(S_)::CLEN; }); }
extern "C" int vrfs_suite_hash_len(vrfs_suite s) { return suite_const(s, [](auto S_) { return (int)decltype(S_)::HLEN; }); }
extern "C" int vrfs_suite_point_enc_len(vrfs_suite s) { return suite_const(s, [](auto S_) { return (int)decltype(S_)::ENC_LEN; }); }

// =================================================================================================
// lincomb launcher
// =================================================================================================
// Kernels on the context's second stream beside the main one: side_fork makes it start after everything enqueued on the main
// stream so far, side_join makes the main stream wait for everything enqueued on it.
static vrfs_status side_fork(vrfs_ctx* ctx) { CU(cudaEventRecord(ctx->ev_fork, ctx->stream)); CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_fork, 0)); return VRFS_OK; }
static vrfs_status side_join(vrfs_ctx* ctx) { CU(cudaEventRecord(ctx->ev_join, ctx->copy_stream)); CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0)); return VRFS_OK; }
// Persistent grid of a lincomb kernel: as many blocks as fit on the GPU at once, but no more than `threads` threads need; each
// thread's window-table slab of `slab_per_thread` bytes in buffer `buf`, and the kernel's work counter behind the slabs (zeroed).
static vrfs_status lincomb_grid(vrfs_ctx* ctx, const void* kernel, size_t threads, size_t slab_per_thread, int buf, cudaStream_t stream,
                                LincombArgs* A, uint32_t* blocks, unsigned block_threads = LINCOMB_THREADS) {
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, (int)block_threads, 0));
  if (per_sm < 1) per_sm = 1;
#ifdef LINCOMB_MAXBLOCKS
  if (per_sm > LINCOMB_MAXBLOCKS) per_sm = LINCOMB_MAXBLOCKS;       // tuning builds: resident threads per SM (the slab scales with them)
#endif
  *blocks = (uint32_t)std::min((size_t)ctx->sms * per_sm, (threads + block_threads - 1) / block_threads);
  const size_t slabs = (size_t)*blocks * block_threads * slab_per_thread;
  void* slab = nullptr;
  ST(ensure(ctx, buf, slabs + 256, &slab));
  A->slab = (uint8_t*)slab;
  A->next_item = reinterpret_cast<uint32_t*>(A->slab + slabs);
  CU(cudaMemsetAsync(A->next_item, 0, sizeof(uint32_t), stream));
  return VRFS_OK;
}
template <int NV, int NF> static const char* lincomb_name() {   // kernel-timing name of k_lincomb<C, NV, NF>
  static constexpr char name[] = {'l', 'i', 'n', 'c', 'o', 'm', 'b', '<', char('0' + NV), ',', char('0' + NF), '>', '\0'}; return name; }
// `side` = true: enqueue on the context's second stream with its own slab, so that two independent linear combinations of a
// small batch (U and V of a verify) run concurrently instead of back to back; the caller forks and joins the streams.
template <class C, int NV, int NF>
static vrfs_status launch_lincomb(vrfs_ctx* ctx, LincombArgs A, bool side = false) {
  if (A.n == 0) return VRFS_OK;
  cudaStream_t stream = side ? ctx->copy_stream : ctx->stream;
  uint32_t blocks = 0;
  ST(lincomb_grid(ctx, (const void*)k_lincomb<C, NV, NF>, A.n, slab_bytes<C>(NV), side ? BUF_SLAB2 : BUF_SLAB, stream, &A, &blocks));
  k_lincomb<C, NV, NF><<<blocks, LINCOMB_THREADS, 0, stream>>>(A);
  LAUNCHED_AS(ctx, (lincomb_name<NV, NF>()));
  return VRFS_OK;
}

template <class C>
static vrfs_status launch_lincomb_verify_pair(vrfs_ctx* ctx, LincombArgs U, LincombArgs V) {
  uint32_t blocks = 0;
  ST(lincomb_grid(ctx, (const void*)k_lincomb_verify_pair<C>, 2 * (size_t)V.n, slab_bytes<C>(2), BUF_SLAB, ctx->stream, &V, &blocks));
  U.slab = V.slab; U.next_item = V.next_item;                         // one slab and one task counter for both combinations
  k_lincomb_verify_pair<C><<<blocks, LINCOMB_THREADS, 0, ctx->stream>>>(U, V);
  LAUNCHED_AS(ctx, "lincomb<1,1>+<2,0>");
  return VRFS_OK;
}
template <class C>
static vrfs_status launch_lincomb_io(vrfs_ctx* ctx, IoArgs A) {
  uint32_t blocks = 0;
  ST(lincomb_grid(ctx, (const void*)k_lincomb_io<C>, A.L.n, slab_bytes<C>(1), BUF_SLAB, ctx->stream, &A.L, &blocks, IO_THREADS));
  k_lincomb_io<C><<<blocks, IO_THREADS, 0, ctx->stream>>>(A);
  LAUNCHED_AS(ctx, "lincomb_io");
  return VRFS_OK;
}

// =================================================================================================
// ietf verify
// =================================================================================================
template <class S>
static vrfs_status ietf_verify_dev(vrfs_ctx* ctx, size_t n, const uint8_t* pk, const uint8_t* input, const uint8_t* output, const uint8_t* c,
                                   const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status = nullptr) {
  typedef typename S::C C;
  void *u = nullptr, *v = nullptr, *valid = nullptr;
  ST(need_tables<S>(ctx));
  ST(ensure(ctx, BUF_W0, n * 96, &u));
  ST(ensure(ctx, BUF_W1, n * 96, &v));
  ST(ensure(ctx, BUF_VALID, n, &valid));
  CU(cudaMemsetAsync(valid, 1, n, ctx->stream));
  LincombArgs A = {};
  A.n = (uint32_t)n;
  A.valid = (uint8_t*)valid;
  // Small batches leave most of the GPU idle and are bound by the latency of one thread's ~4 100 products: run U and V side by
  // side on two streams (both grids fit at once).  Large batches fill the GPU either way and stay on one stream.
  // (overlapping the two launches of a LARGE batch the same way was measured at +0.3 %: not worth losing per-kernel timing)
  const bool split = n <= (size_t)ctx->sms * VRFS_SPLIT_ITEMS_PER_SM;
  const uint32_t cbits = S::CLEN < 32 ? 8u * S::CLEN : 0u;     // a CHALLENGE_LEN-byte challenge: half of its windows are empty
  // mid-size batches (between the two-stream case and VRFS_PAIR_WAVES resident waves): one grid for both combinations
  if (!split && VRFS_PAIR_WAVES > 0 && n < (size_t)ctx->sms * LINCOMB_THREADS * LINCOMB_MINBLOCKS * VRFS_PAIR_WAVES) {
    LincombArgs U = A, V = A;
    U.var[0] = {pk, 64, c, 32, 1, cbits};
    U.fix[0] = {s, 32, 0, ctx->fixtab[S::ID][0]};
    U.out_xyz = (uint32_t*)u;
    V.var[0] = {input, 64, s, 32, 0, 0};
    V.var[1] = {output, 64, c, 32, 1, cbits};
    V.out_xyz = (uint32_t*)v;
    ST((launch_lincomb_verify_pair<C>(ctx, U, V)));
    k_ietf_verify_finish<S><<<(unsigned)((n + 128 * FINISH_K - 1) / (128 * FINISH_K)), 128, 0, ctx->stream>>>((uint32_t)n, pk, input, output, c, (const uint32_t*)u,
                                                                                  (const uint32_t*)v, ad, ad_off, (const uint8_t*)valid, out_ok, out_status);
    LAUNCHED_AS(ctx, "ietf_verify_finish");
    return VRFS_OK;
  }
  // U = s*G - c*Y
  A.var[0] = {pk, 64, c, 32, 1, cbits};
  A.fix[0] = {s, 32, 0, ctx->fixtab[S::ID][0]};
  A.out_xyz = (uint32_t*)u;
  if (split) ST(side_fork(ctx));   // the side stream starts after the inputs and the memset of `valid`
  ST((launch_lincomb<C, 1, 1>(ctx, A, split)));
  // V = s*I - c*O
  A.var[0] = {input, 64, s, 32, 0, 0};
  A.var[1] = {output, 64, c, 32, 1, cbits};
  A.out_xyz = (uint32_t*)v;
  ST((launch_lincomb<C, 2, 0>(ctx, A)));
  if (split) ST(side_join(ctx));
  k_ietf_verify_finish<S><<<(unsigned)((n + 128 * FINISH_K - 1) / (128 * FINISH_K)), 128, 0, ctx->stream>>>((uint32_t)n, pk, input, output, c, (const uint32_t*)u,
                                                                                (const uint32_t*)v, ad, ad_off, (const uint8_t*)valid, out_ok, out_status);
  LAUNCHED_AS(ctx, "ietf_verify_finish");
  return VRFS_OK;
}

extern "C" vrfs_status vrfs_ietf_verify_batch_dev(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pk, const uint8_t* input,
                                                  const uint8_t* output, const uint8_t* c, const uint8_t* s, const uint8_t* ad,
                                                  const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!pk || !input || !output || !c || !s || !out_ok || (ad && !ad_off)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (!aligned16(pk) || !aligned16(input) || !aligned16(output) || !aligned16(c) || !aligned16(s)) return fail(ctx, VRFS_BAD_ARG, "device buffers must be 16-byte aligned");
  ST(begin_call(ctx, suite, n));
  return with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return ietf_verify_dev<S>(ctx, n, pk, input, output, c, s, ad, ad_off, out_ok, out_status); });
}

// host -> device staging of one input; returns the device pointer
static vrfs_status stage_in(vrfs_ctx* ctx, int which, const void* host, size_t bytes, const uint8_t** dev) {
  void* d = nullptr;
  ST(ensure(ctx, which, bytes, &d));
  if (bytes) CU(cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
  // kernel timing: the first kernel's interval starts after the last input copy, not at the start of the call
  if (ctx->timing && ctx->tev[0] && ctx->n_timed == 0) CU(cudaEventRecord(ctx->tev[0], ctx->stream));
  *dev = (const uint8_t*)d;
  return VRFS_OK;
}
static vrfs_status stage_ad(vrfs_ctx* ctx, size_t n, const uint8_t* ad, const uint64_t* ad_off, const uint8_t** d_ad, const uint64_t** d_off) {
  *d_ad = nullptr; *d_off = nullptr;
  if (!ad_off) return VRFS_OK;
  for (size_t i = 0; i < n; i++) if (ad_off[i + 1] < ad_off[i]) return fail(ctx, VRFS_BAD_ARG, "offsets must be non-decreasing");
  if (ad_off[n] > ad_off[0] && !ad) return fail(ctx, VRFS_BAD_ARG, "null data buffer with non-empty offsets");
  // only the bytes these n items refer to travel (a shard of a larger batch passes ad_off + lo: absolute offsets into `ad`);
  // the device pointer is biased so that the kernels keep indexing with the absolute offsets
  const uint8_t *o = nullptr, *base = nullptr;
  ST(stage_in(ctx, BUF_AD, ad ? ad + ad_off[0] : nullptr, (size_t)(ad_off[n] - ad_off[0]), &base));
  *d_ad = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(base) - (uintptr_t)ad_off[0]);
  ST(stage_in(ctx, BUF_OFF, ad_off, (n + 1) * sizeof(uint64_t), &o));
  *d_off = (const uint64_t*)o;
  return VRFS_OK;
}
// variable-length items (h2c data): validated offsets + bytes -> device
static vrfs_status stage_var(vrfs_ctx* ctx, int buf_data, int buf_off, size_t n, const uint8_t* data, const uint64_t* off, const uint8_t** d_data, const uint64_t** d_off) {
  for (size_t i = 0; i < n; i++) if (off[i + 1] < off[i]) return fail(ctx, VRFS_BAD_ARG, "offsets must be non-decreasing");
  if (off[n] > 0 && !data) return fail(ctx, VRFS_BAD_ARG, "null data buffer with non-empty offsets");
  const uint8_t* o = nullptr;
  ST(stage_in(ctx, buf_data, data, (size_t)off[n], d_data));
  ST(stage_in(ctx, buf_off, off, (n + 1) * sizeof(uint64_t), &o));
  *d_off = (const uint64_t*)o;
  return VRFS_OK;
}

// =================================================================================================
// measurement helper
// =================================================================================================
extern "C" vrfs_status vrfs_measure_mac32_peak(vrfs_ctx* ctx, int variant, double* out_mac_per_s, double* out_sm_mhz_est) {
  if (!ctx || !out_mac_per_s) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  CU(cudaSetDevice(ctx->device));
  const int threads = 256, blocks = ctx->sms * 8;
  void *out = nullptr, *cyc = nullptr;
  ST(ensure(ctx, BUF_W0, (size_t)threads * blocks * 4, &out));
  ST(ensure(ctx, BUF_W1, 64, &cyc));
  const bool field_mul = (variant == 2 || variant == 3);
  int iters = field_mul ? 64 : 4096;
  double macs_per_thread_iter = field_mul ? 32.0 * 136.0 : 32.0;   // field products are counted as 136 MAC32 (the saturated 8-limb model) in every representation
  float ms = 0;
  for (int rep = 0; rep < 3; rep++) {
    CU(cudaEventRecord(ctx->ev0, ctx->stream));
    switch (variant) {
      case 0: k_mac_bench<0><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 1: k_mac_bench<1><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 2: k_mac_bench<2><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 3: k_mac_bench<3><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 4: k_mac_bench<4><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 5: k_mac_bench<5><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 6: k_mac_bench<6><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      case 9: k_mac_bench<9><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, (unsigned long long*)cyc); break;
      default: return fail(ctx, VRFS_BAD_ARG, "unknown variant %d", variant);
    }
    LAUNCHED(ctx);
    CU(cudaEventRecord(ctx->ev1, ctx->stream));
    CU(cudaEventSynchronize(ctx->ev1));
    CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  }
  unsigned long long cycles = 0;
  CU(cudaMemcpy(&cycles, cyc, sizeof cycles, cudaMemcpyDeviceToHost));
  *out_mac_per_s = macs_per_thread_iter * iters * (double)threads * blocks / (ms * 1e-3);
  if (out_sm_mhz_est) *out_sm_mhz_est = (double)cycles / (ms * 1e-3) / 1e6;
  return VRFS_OK;
}


// =================================================================================================
// per-item kernels of the remaining twisted-Edwards entry points (one thread per item)
// =================================================================================================
#define ITEM_THREADS 128
#define ITEM_INDEX(n) uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= (n)) return
#define VAR_SLICE(buf, off, i, ptr, len) const uint8_t* ptr = (buf) ? (buf) + (off)[i] : nullptr; uint32_t len = (buf) ? (uint32_t)((off)[(i) + 1] - (off)[i]) : 0u
static inline unsigned item_blocks(size_t n) { return (unsigned)((n + ITEM_THREADS - 1) / ITEM_THREADS); }

template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_nonce(uint32_t n, const uint8_t* sk, const uint8_t* input, uint8_t* out_k) {
  ITEM_INDEX(n);
  nonce_item<S>(out_k + (size_t)32 * i, sk + (size_t)32 * i, input + (size_t)64 * i);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_ietf_prove_finish(uint32_t n, const uint8_t* sk, const uint8_t* k, const uint8_t* input, const uint8_t* output,
                                                                                        const uint32_t* y, const uint32_t* kg, const uint32_t* ki, const uint8_t* ad, const uint64_t* ad_off,
                                                                                        const uint8_t* valid, const uint32_t* zinv, uint8_t* out_c, uint8_t* out_s) {
  ITEM_INDEX(n);
  VAR_SLICE(ad, ad_off, i, a, alen);
  uint8_t* oc = out_c + (size_t)32 * i; uint8_t* os = out_s + (size_t)32 * i;
  if (!valid[i]) { for (int j = 0; j < 32; j++) { oc[j] = 0; os[j] = 0; } return; }
  ietf_prove_finish_item<S>(oc, os, sk + (size_t)32 * i, k + (size_t)32 * i, input + (size_t)64 * i, output + (size_t)64 * i,
                            y + (size_t)24 * i, kg + (size_t)24 * i, ki + (size_t)24 * i, a, alen, zinv + (size_t)8 * i);
}
// one field inversion per ZINV_K items: zinv[i] = 1 / (product of the Z's of item i's NP projective points)
#define ZINV_K 8
template <class C, int NP> __global__ void __launch_bounds__(128) k_zinv(uint32_t n, const uint32_t* p0, const uint32_t* p1, const uint32_t* p2, uint32_t* zinv) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  if (t >= n) return;
  const uint32_t* pts[3] = {p0, p1, p2};
  zinv_batched<C, NP, ZINV_K>(n, t, stride, pts, zinv);
}
// projective -> affine ABI bytes, one point per item (Secret::output, Public)
template <class C> __global__ void __launch_bounds__(ITEM_THREADS) k_to_affine(uint32_t n, const uint32_t* xyz, const uint8_t* valid, const uint32_t* zinv, uint8_t* out) {
  ITEM_INDEX(n);
  uint8_t* o = out + (size_t)64 * i;
  if (valid && !valid[i]) { for (int j = 0; j < 64; j++) o[j] = 0; return; }
  typename C::F ax[1], ay[1];
  const uint32_t* pp[1] = {xyz + (size_t)24 * i};
  to_affine_shared<C, 1>(ax, ay, pp, zinv + (size_t)8 * i);
  store_affine_bytes<C>(o, ax[0], ay[0]);
}
// Secret::from_seed: sk = LE(H(seed)) mod r
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_secret_from_seed(uint32_t n, const uint8_t* seeds, const uint64_t* off, uint8_t* out_sk) {
  ITEM_INDEX(n);
  VAR_SLICE(seeds, off, i, p, len);
  typename S::H h; h.init(); h.update(p, len);
  uint8_t d[S::HLEN]; h.final(d);
  uint32_t k[8];
  hash_to_scalar<typename S::C>(k, d, S::HLEN, false);
  store_le<8>(out_sk + (size_t)32 * i, k);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_point_to_hash(uint32_t n, const uint8_t* pts, uint8_t* out) {
  ITEM_INDEX(n);
  typedef typename S::C C;
  typename C::F x, y;
  bool inf = false;
  uint8_t* o = out + (size_t)S::HLEN * i;
  if (!load_affine<C>(x, y, &inf, pts + (size_t)64 * i) || inf) { for (int j = 0; j < S::HLEN; j++) o[j] = 0; return; }
  uint8_t enc[S::ENC_LEN];
  encode_point_bytes<S>(enc, pts + (size_t)64 * i);
  suite_point_to_hash<S>(o, enc);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_point_encode(uint32_t n, const uint8_t* pts, uint8_t* out) {
  ITEM_INDEX(n);
  typedef typename S::C C;
  typename C::F x, y;
  bool inf = false;
  uint8_t* o = out + (size_t)S::ENC_LEN * i;
  if (!load_affine<C>(x, y, &inf, pts + (size_t)64 * i) || inf) { for (int j = 0; j < S::ENC_LEN; j++) o[j] = 0; return; }
  encode_point_bytes<S>(o, pts + (size_t)64 * i);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_point_decode(uint32_t n, const uint8_t* enc, uint8_t* out, uint8_t* out_ok) {
  ITEM_INDEX(n);
  typedef typename S::C C;
  typename C::F x, y;
  uint8_t* o = out + (size_t)64 * i;
  bool ok = decode_point<S>(x, y, enc + (size_t)S::ENC_LEN * i);
  out_ok[i] = ok;
  if (ok) store_affine_bytes<C>(o, x, y); else for (int j = 0; j < 64; j++) o[j] = 0;
}
// Suite::data_to_point (K6)
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_data_to_point(uint32_t n, const uint8_t* data, const uint64_t* off, uint32_t* out_xyz, uint8_t* out_ok) {
  ITEM_INDEX(n);
  typedef typename S::C C;
  VAR_SLICE(data, off, i, p, len);
  typename C::F X, Y, Z;
  bool ok;
  if constexpr (C::HAS_GLV) { TEPoint<C> P; band_h2c_ell2(P, p, len); ok = true; X = P.X; Y = P.Y; Z = P.Z; }
  else { typename Grp<C>::Pt P; ok = h2c_tai<S>(P, p, len); X = P.X; Y = P.Y; Z = P.Z; }
  out_ok[i] = ok;
  if (!ok) { X = C::F::zero(); Y = C::F::one(); Z = C::F::one(); }
  store_fp_xyz(out_xyz + (size_t)24 * i, X, Y, Z);      // projective: the inversion is shared by 8 items (k_zinv + k_to_affine)
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_pedersen_prove_prep(uint32_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* ad, const uint64_t* ad_off,
                                                                                          uint8_t* b, uint8_t* k, uint8_t* kb) {
  ITEM_INDEX(n);
  VAR_SLICE(ad, ad_off, i, a, alen);
  pedersen_prove_prep_item<S>(b + (size_t)32 * i, k + (size_t)32 * i, kb + (size_t)32 * i, sk + (size_t)32 * i, input + (size_t)64 * i, a, alen);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_pedersen_prove_finish(uint32_t n, const uint8_t* sk, const uint8_t* b, const uint8_t* k, const uint8_t* kb,
                                                                                            const uint8_t* input, const uint8_t* output, const uint32_t* yb, const uint32_t* r, const uint32_t* okp,
                                                                                            const uint8_t* ad, const uint64_t* ad_off, const uint8_t* valid, const uint32_t* zinv, uint8_t* proof, uint8_t* blinding) {
  ITEM_INDEX(n);
  VAR_SLICE(ad, ad_off, i, a, alen);
  uint8_t* pr = proof + (size_t)256 * i; uint8_t* bl = blinding + (size_t)32 * i;
  if (!valid[i]) { for (int j = 0; j < 256; j++) pr[j] = 0; for (int j = 0; j < 32; j++) bl[j] = 0; return; }
  pedersen_prove_finish_item<S>(pr, sk + (size_t)32 * i, b + (size_t)32 * i, k + (size_t)32 * i, kb + (size_t)32 * i, input + (size_t)64 * i,
                                output + (size_t)64 * i, yb + (size_t)24 * i, r + (size_t)24 * i, okp + (size_t)24 * i, a, alen, zinv + (size_t)8 * i);
  for (int j = 0; j < 32; j++) bl[j] = b[(size_t)32 * i + j];
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_pedersen_verify_prep(uint32_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof,
                                                                                           const uint8_t* ad, const uint64_t* ad_off, uint8_t* c, uint8_t* valid) {
  ITEM_INDEX(n);
  VAR_SLICE(ad, ad_off, i, a, alen);
  if (!pedersen_verify_prep_item<S>(c + (size_t)32 * i, input + (size_t)64 * i, output + (size_t)64 * i, proof + (size_t)256 * i, a, alen)) valid[i] = 0;
}
// Ok + c*O == s*I  and  R + c*Yb == s*G + sb*B, given T1 = s*I - c*O and T2 = s*G + sb*B - c*Yb (projective)
template <class C> __global__ void __launch_bounds__(ITEM_THREADS) k_pedersen_verify_finish(uint32_t n, const uint8_t* proof, const uint32_t* t1, const uint32_t* t2,
                                                                                             const uint8_t* valid, uint8_t* out_ok, uint8_t* out_status) {
  ITEM_INDEX(n);
  const uint8_t* pr = proof + (size_t)256 * i;
  const int e1 = proj_vs_affine_bytes<C>(t1 + (size_t)24 * i, pr + 128), e2 = proj_vs_affine_bytes<C>(t2 + (size_t)24 * i, pr + 64);
  const bool good = e1 == 2 && e2 == 2 && valid[i];
  out_ok[i] = (uint8_t)good;
  // `valid` is cleared by the linear combinations for I, O, Yb that are no curve points and by the prep kernel for identities;
  // R and Ok are validated here
  if (out_status) out_status[i] = (uint8_t)(good ? ITEM_OK : (!valid[i] || e1 == 0 || e2 == 0) ? ITEM_INVALID_DATA : ITEM_VERIFICATION_FAILURE);
}

// =================================================================================================
// host-side plumbing shared by the entry points below
// =================================================================================================
static vrfs_status stage_out(vrfs_ctx* ctx, int which, size_t bytes, uint8_t** dev) {
  void* d = nullptr;
  ST(ensure(ctx, which, bytes, &d));
  *dev = (uint8_t*)d;
  return VRFS_OK;
}
static vrfs_status copy_out(vrfs_ctx* ctx, void* host, const void* dev, size_t bytes) {
  if (bytes) CU(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return VRFS_OK;
}
static vrfs_status finish_call(vrfs_ctx* ctx) {
  CU(cudaStreamSynchronize(ctx->stream));
  return VRFS_OK;
}
static vrfs_status fresh_valid(vrfs_ctx* ctx, size_t n, uint8_t** valid) {
  void* v = nullptr;
  ST(ensure(ctx, BUF_VALID, n, &v));
  CU(cudaMemsetAsync(v, 1, n, ctx->stream));
  *valid = (uint8_t*)v;
  return VRFS_OK;
}
template <class S> static const void* fixtab(vrfs_ctx* ctx, int which) { return ctx->fixtab[S::ID][which]; }   // after need_tables<S>
// key material on the device: remembered per buffer, zeroed by the outermost CallGuard
static void mark_secret(vrfs_ctx* ctx, int which, size_t bytes) { if (ctx->buf[which].secret_bytes < bytes) ctx->buf[which].secret_bytes = bytes; }
static vrfs_status stage_secret(vrfs_ctx* ctx, int which, const void* host, size_t bytes, const uint8_t** dev) {
  mark_secret(ctx, which, bytes);
  return stage_in(ctx, which, host, bytes, dev);
}
// Host buffers of a large batch call travel in PIECES on the copy stream: one resident wave of the lincomb grid first, then the
// rest in up to max_pieces - 1 runs of whole waves.  Piece k's kernels wait only for piece k's inputs, so all but the first
// ~20 MB of the input transfer hides behind arithmetic (pinned host memory; pageable memory still works, the copies then
// serialise inside the driver), and piece k's results go back to the host while piece k + 1 computes (pieces_copy_out) - what
// matters for the prove calls, whose outputs are 64-288 B per item.
struct HostIn { int buf; const void* host; size_t stride; bool secret; uint8_t* dev; };
struct HostOut { void* host; const uint8_t* dev; size_t stride; };
struct Pieces { size_t cut[VRFS_HOST_PIECES + 1]; int count; };
static vrfs_status stage_in_pieces(vrfs_ctx* ctx, size_t n, HostIn* in, int nin, Pieces* pc, int max_pieces) {
  const size_t wave = (size_t)ctx->sms * LINCOMB_MINBLOCKS * LINCOMB_THREADS;
  pc->cut[0] = 0; pc->cut[1] = n; pc->count = 1;
  if (n > 3 * wave && max_pieces >= 2) {
    if (max_pieces > VRFS_HOST_PIECES) max_pieces = VRFS_HOST_PIECES;
    const size_t rest_waves = (n - wave + wave - 1) / wave;
    const size_t q = rest_waves < (size_t)(max_pieces - 1) ? rest_waves : (size_t)(max_pieces - 1);
    const size_t per = (rest_waves + q - 1) / q * wave;
    pc->cut[1] = wave;
    while (pc->cut[pc->count] < n) {
      const size_t next = pc->cut[pc->count] + per;
      pc->count++;
      pc->cut[pc->count] = next < n ? next : n;
    }
  }
  for (int j = 0; j < nin; j++) {
    void* d = nullptr;
    ST(ensure(ctx, in[j].buf, n * in[j].stride, &d));
    in[j].dev = (uint8_t*)d;
    if (in[j].secret) mark_secret(ctx, in[j].buf, n * in[j].stride);
  }
  for (int k = 0; k < pc->count; k++) {
    const size_t o = pc->cut[k], m = pc->cut[k + 1] - pc->cut[k];
    for (int j = 0; j < nin; j++)
      CU(cudaMemcpyAsync(in[j].dev + o * in[j].stride, (const uint8_t*)in[j].host + o * in[j].stride, m * in[j].stride, cudaMemcpyHostToDevice, ctx->copy_stream));
    CU(cudaEventRecord(ctx->ev_in[k], ctx->copy_stream));
  }
  return VRFS_OK;
}
static vrfs_status piece_ready(vrfs_ctx* ctx, int k) {
  CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[k], 0));
  // kernel timing: the first kernel's interval starts after its inputs arrived, not at the start of the call
  if (ctx->timing && ctx->tev[0] && ctx->n_timed == 0) CU(cudaEventRecord(ctx->tev[0], ctx->stream));
  return VRFS_OK;
}
// results of piece k back to the host on the copy stream, behind the kernels of piece k; the last piece makes the main stream
// wait for every copy, so that finish_call (and the wipe of secret buffers after it) sees them all done
static vrfs_status pieces_copy_out(vrfs_ctx* ctx, const Pieces& pc, int k, const HostOut* out, int nout) {
  const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
  CU(cudaEventRecord(ctx->ev_out[k], ctx->stream));
  CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_out[k], 0));
  for (int j = 0; j < nout; j++)
    CU(cudaMemcpyAsync((uint8_t*)out[j].host + o * out[j].stride, out[j].dev + o * out[j].stride, m * out[j].stride, cudaMemcpyDeviceToHost, ctx->copy_stream));
  if (k == pc.count - 1) {
    CU(cudaEventRecord(ctx->ev_out[k], ctx->copy_stream));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_out[k], 0));
  }
  return VRFS_OK;
}
// batched inversion of the Z coordinates of NP projective results per item (k_zinv): returns the device array of n x 8 words
template <class C, int NP> static vrfs_status launch_zinv(vrfs_ctx* ctx, size_t n, const void* p0, const void* p1, const void* p2, const uint32_t** out) {
  void* z = nullptr;
  ST(ensure(ctx, BUF_ZINV, n * 32, &z));
  const size_t threads = (n + ZINV_K - 1) / ZINV_K;
  k_zinv<C, NP><<<(unsigned)((threads + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)p0, (const uint32_t*)p1, (const uint32_t*)p2, (uint32_t*)z);
  LAUNCHED_AS(ctx, "zinv");
  *out = (const uint32_t*)z;
  return VRFS_OK;
}
// Suite::data_to_point: hash-to-curve kernel (projective) + batched inversion + affine ABI bytes (zeros where no point was found)
template <class S> static vrfs_status data_to_point_dev(vrfs_ctx* ctx, size_t n, const uint8_t* data, const uint64_t* off, uint8_t* out_pts, uint8_t* out_ok) {
  typedef typename S::C C;
  void* xyz = nullptr;
  ST(ensure(ctx, BUF_W0, n * 96, &xyz));
  k_data_to_point<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, data, off, (uint32_t*)xyz, out_ok);
  LAUNCHED_AS(ctx, "data_to_point");
  const uint32_t* zinv = nullptr;
  ST((launch_zinv<C, 1>(ctx, n, xyz, nullptr, nullptr, &zinv)));
  k_to_affine<C><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)xyz, out_ok, zinv, out_pts);
  LAUNCHED_AS(ctx, "to_affine");
  return VRFS_OK;
}

// ---- ietf verify (host buffers) ------------------------------------------------------------
// Everything enqueued and nothing waited for (the multi-device context enqueues one of these per GPU before it waits for any):
// the inputs travel in two pieces (stage_in_pieces), the 1 B/item of verdicts return on the main stream after the last piece.
static vrfs_status ietf_verify_host_enqueue(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pk, const uint8_t* input, const uint8_t* output,
                                            const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!pk || !input || !output || !c || !s || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_ok, *d_st = nullptr;
  // ad and the result buffers first: a buffer that grows is reallocated, which waits for the copies already in flight
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  HostIn in[5] = {{BUF_IN0, pk, 64, false, nullptr}, {BUF_IN1, input, 64, false, nullptr}, {BUF_IN2, output, 64, false, nullptr},
                  {BUF_IN3, c, 32, false, nullptr}, {BUF_IN4, s, 32, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 5, &pc, 2));
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_verify_dev<S>(ctx, m, in[0].dev + o * 64, in[1].dev + o * 64, in[2].dev + o * 64, in[3].dev + o * 32, in[4].dev + o * 32, d_ad,
                                d_off ? d_off + o : nullptr, d_ok + o, d_st ? d_st + o : nullptr); }));
  }
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ietf_verify_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pk, const uint8_t* input,
                                              const uint8_t* output, const uint8_t* c, const uint8_t* s, const uint8_t* ad,
                                              const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  ST(ietf_verify_host_enqueue(ctx, suite, n, pk, input, output, c, s, ad, ad_off, out_ok, out_status));
  return finish_call(ctx);
}

// ---- ietf prove -----------------------------------------------------------------------------
template <class S>
static vrfs_status ietf_prove_dev(vrfs_ctx* ctx, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output, const uint8_t* ad,
                                  const uint64_t* ad_off, uint8_t* out_c, uint8_t* out_s) {
  typedef typename S::C C;
  void *k = nullptr, *y = nullptr, *kg = nullptr, *ki = nullptr;
  uint8_t* valid = nullptr;
  ST(need_tables<S>(ctx));
  ST(ensure(ctx, BUF_W0, n * 32, &k)); ST(ensure(ctx, BUF_W1, n * 96, &y)); ST(ensure(ctx, BUF_W2, n * 96, &kg)); ST(ensure(ctx, BUF_W3, n * 96, &ki));
  mark_secret(ctx, BUF_W0, n * 32);                      // the nonces k
  ST(fresh_valid(ctx, n, &valid));
  k_nonce<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sk, input, (uint8_t*)k);
  LAUNCHED_AS(ctx, "nonce");
  LincombArgs A = {};
  A.n = (uint32_t)n; A.valid = valid;
  A.fix[0] = {sk, 32, 0, fixtab<S>(ctx, 0)}; A.out_xyz = (uint32_t*)y;
  ST((launch_lincomb<C, 0, 1>(ctx, A)));
  A.fix[0] = {(const uint8_t*)k, 32, 0, fixtab<S>(ctx, 0)}; A.out_xyz = (uint32_t*)kg;
  ST((launch_lincomb<C, 0, 1>(ctx, A)));
  A.var[0] = {input, 64, (const uint8_t*)k, 32, 0}; A.out_xyz = (uint32_t*)ki;
  ST((launch_lincomb<C, 1, 0>(ctx, A)));
  const uint32_t* zinv = nullptr;
  ST((launch_zinv<C, 3>(ctx, n, y, kg, ki, &zinv)));
  k_ietf_prove_finish<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sk, (const uint8_t*)k, input, output, (const uint32_t*)y,
                                                                           (const uint32_t*)kg, (const uint32_t*)ki, ad, ad_off, valid, zinv, out_c, out_s);
  LAUNCHED_AS(ctx, "ietf_prove_finish");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ietf_prove_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output,
                                             const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_c, uint8_t* out_s) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !input || !output || !out_c || !out_s) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_c, *d_s;
  HostIn in[3] = {{BUF_IN0, sk, 32, true, nullptr}, {BUF_IN1, input, 64, false, nullptr}, {BUF_IN2, output, 64, false, nullptr}};
  Pieces pc;   // two pieces: every further piece costs ~1 % in kernel tails, more than hiding the rest of the 64 B/item of results returns
  ST(stage_in_pieces(ctx, n, in, 3, &pc, 2));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n * 32, &d_c)); ST(stage_out(ctx, BUF_OUT1, n * 32, &d_s));
  const HostOut out[2] = {{out_c, d_c, 32}, {out_s, d_s, 32}};
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_prove_dev<S>(ctx, m, in[0].dev + o * 32, in[1].dev + o * 64, in[2].dev + o * 64, d_ad, d_off ? d_off + o : nullptr, d_c + o * 32, d_s + o * 32); }));
    ST(pieces_copy_out(ctx, pc, k, out, 2));
  }
  return finish_call(ctx);
}

// ---- Secret::output, Secret::from_seed, nonce, point_to_hash, codec, data_to_point ------------
template <class S> static vrfs_status output_dev(vrfs_ctx* ctx, size_t n, const uint8_t* sk, const uint8_t* input, uint8_t* out) {
  typedef typename S::C C;
  void* o = nullptr; uint8_t* valid = nullptr;
  ST(ensure(ctx, BUF_W0, n * 96, &o)); ST(fresh_valid(ctx, n, &valid));
  LincombArgs A = {};
  A.n = (uint32_t)n; A.valid = valid; A.var[0] = {input, 64, sk, 32, 0}; A.out_xyz = (uint32_t*)o;
  ST((launch_lincomb<C, 1, 0>(ctx, A)));
  const uint32_t* zinv = nullptr;
  ST((launch_zinv<C, 1>(ctx, n, o, nullptr, nullptr, &zinv)));
  k_to_affine<C><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)o, valid, zinv, out);
  LAUNCHED_AS(ctx, "to_affine");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_output_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* input, uint8_t* out_output) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !input || !out_output) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t *d_sk, *d_in; uint8_t* d_o;
  ST(stage_secret(ctx, BUF_IN0, sk, n * 32, &d_sk)); ST(stage_in(ctx, BUF_IN1, input, n * 64, &d_in)); ST(stage_out(ctx, BUF_OUT0, n * 64, &d_o));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return output_dev<S>(ctx, n, d_sk, d_in, d_o); }));
  ST(copy_out(ctx, out_output, d_o, n * 64));
  return finish_call(ctx);
}
template <class S> static vrfs_status from_seed_dev(vrfs_ctx* ctx, size_t n, const uint8_t* seeds, const uint64_t* off, uint8_t* out_sk, uint8_t* out_pk) {
  typedef typename S::C C;
  k_secret_from_seed<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, seeds, off, out_sk);
  LAUNCHED_AS(ctx, "secret_from_seed");
  if (!out_pk) return VRFS_OK;
  ST(need_tables<S>(ctx));
  void* o = nullptr;
  ST(ensure(ctx, BUF_W0, n * 96, &o));
  LincombArgs A = {};
  A.n = (uint32_t)n; A.fix[0] = {out_sk, 32, 0, fixtab<S>(ctx, 0)}; A.out_xyz = (uint32_t*)o;
  ST((launch_lincomb<C, 0, 1>(ctx, A)));
  const uint32_t* zinv = nullptr;
  ST((launch_zinv<C, 1>(ctx, n, o, nullptr, nullptr, &zinv)));
  k_to_affine<C><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)o, nullptr, zinv, out_pk);
  LAUNCHED_AS(ctx, "to_affine");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_secret_from_seed_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* seeds, const uint64_t* seed_off,
                                                   uint8_t* out_sk, uint8_t* out_pk) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!seed_off || !out_sk) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_seeds; const uint64_t* d_off; uint8_t *d_sk, *d_pk = nullptr;
  ST(stage_ad(ctx, n, seeds, seed_off, &d_seeds, &d_off));
  mark_secret(ctx, BUF_AD, (size_t)(seed_off[n] - seed_off[0]));
  ST(stage_out(ctx, BUF_OUT0, n * 32, &d_sk));
  mark_secret(ctx, BUF_OUT0, n * 32);
  if (out_pk) ST(stage_out(ctx, BUF_OUT1, n * 64, &d_pk));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return from_seed_dev<S>(ctx, n, d_seeds, d_off, d_sk, d_pk); }));
  ST(copy_out(ctx, out_sk, d_sk, n * 32));
  if (out_pk) ST(copy_out(ctx, out_pk, d_pk, n * 64));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_nonce_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* input, uint8_t* out_k) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !input || !out_k) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t *d_sk, *d_in; uint8_t* d_k;
  ST(stage_secret(ctx, BUF_IN0, sk, n * 32, &d_sk)); ST(stage_in(ctx, BUF_IN1, input, n * 64, &d_in)); ST(stage_out(ctx, BUF_OUT0, n * 32, &d_k));
  mark_secret(ctx, BUF_OUT0, n * 32);
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; k_nonce<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, d_sk, d_in, d_k); return VRFS_OK; }));
  LAUNCHED_AS(ctx, "nonce");
  ST(copy_out(ctx, out_k, d_k, n * 32));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_point_to_hash_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pts, uint8_t* out_hash) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!pts || !out_hash) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_p; uint8_t* d_h;
  const size_t hl = (size_t)vrfs_suite_hash_len(suite);
  ST(stage_in(ctx, BUF_IN0, pts, n * 64, &d_p)); ST(stage_out(ctx, BUF_OUT0, n * hl, &d_h));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; k_point_to_hash<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, d_p, d_h); return VRFS_OK; }));
  LAUNCHED_AS(ctx, "point_to_hash");
  ST(copy_out(ctx, out_hash, d_h, n * hl));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_point_encode_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pts, uint8_t* out_enc) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!pts || !out_enc) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_p; uint8_t* d_e;
  const size_t el = (size_t)vrfs_suite_point_enc_len(suite);
  ST(stage_in(ctx, BUF_IN0, pts, n * 64, &d_p)); ST(stage_out(ctx, BUF_OUT0, n * el, &d_e));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; k_point_encode<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, d_p, d_e); return VRFS_OK; }));
  LAUNCHED_AS(ctx, "point_encode");
  ST(copy_out(ctx, out_enc, d_e, n * el));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_point_decode_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* enc, uint8_t* out_pts, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!enc || !out_pts || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_e; uint8_t *d_p, *d_ok;
  const size_t el = (size_t)vrfs_suite_point_enc_len(suite);
  ST(stage_in(ctx, BUF_IN0, enc, n * el, &d_e)); ST(stage_out(ctx, BUF_OUT0, n * 64, &d_p)); ST(stage_out(ctx, BUF_OUT1, n, &d_ok));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; k_point_decode<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, d_e, d_p, d_ok); return VRFS_OK; }));
  LAUNCHED_AS(ctx, "point_decode");
  ST(copy_out(ctx, out_pts, d_p, n * 64)); ST(copy_out(ctx, out_ok, d_ok, n));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_data_to_point_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* data, const uint64_t* data_off,
                                                uint8_t* out_pts, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!data_off || !out_pts || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_d; const uint64_t* d_off; uint8_t *d_p, *d_ok;
  ST(stage_ad(ctx, n, data, data_off, &d_d, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n * 64, &d_p)); ST(stage_out(ctx, BUF_OUT1, n, &d_ok));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return data_to_point_dev<S>(ctx, n, d_d, d_off, d_p, d_ok); }));
  ST(copy_out(ctx, out_pts, d_p, n * 64)); ST(copy_out(ctx, out_ok, d_ok, n));
  return finish_call(ctx);
}

// ---- pedersen ---------------------------------------------------------------------------------
template <class S>
static vrfs_status pedersen_prove_dev(vrfs_ctx* ctx, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output, const uint8_t* ad,
                                      const uint64_t* ad_off, uint8_t* proof, uint8_t* blinding) {
  typedef typename S::C C;
  void *sc = nullptr, *yb = nullptr, *r = nullptr, *okp = nullptr;
  uint8_t* valid = nullptr;
  ST(need_tables<S>(ctx));
  ST(ensure(ctx, BUF_W0, n * 96, &sc)); ST(ensure(ctx, BUF_W1, n * 96, &yb)); ST(ensure(ctx, BUF_W2, n * 96, &r)); ST(ensure(ctx, BUF_W3, n * 96, &okp));
  mark_secret(ctx, BUF_W0, n * 96);                      // blinding factor b and the nonces k, kb
  ST(fresh_valid(ctx, n, &valid));
  uint8_t *b = (uint8_t*)sc, *k = b + n * 32, *kb = k + n * 32;
  k_pedersen_prove_prep<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sk, input, ad, ad_off, b, k, kb);
  LAUNCHED_AS(ctx, "pedersen_prove_prep");
  LincombArgs A = {};
  A.n = (uint32_t)n; A.valid = valid;
  A.fix[0] = {sk, 32, 0, fixtab<S>(ctx, 0)}; A.fix[1] = {b, 32, 0, fixtab<S>(ctx, 1)}; A.out_xyz = (uint32_t*)yb;
  ST((launch_lincomb<C, 0, 2>(ctx, A)));
  A.fix[0] = {k, 32, 0, fixtab<S>(ctx, 0)}; A.fix[1] = {kb, 32, 0, fixtab<S>(ctx, 1)}; A.out_xyz = (uint32_t*)r;
  ST((launch_lincomb<C, 0, 2>(ctx, A)));
  A.var[0] = {input, 64, k, 32, 0}; A.out_xyz = (uint32_t*)okp;
  ST((launch_lincomb<C, 1, 0>(ctx, A)));
  const uint32_t* zinv = nullptr;
  ST((launch_zinv<C, 3>(ctx, n, yb, r, okp, &zinv)));
  k_pedersen_prove_finish<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sk, b, k, kb, input, output, (const uint32_t*)yb, (const uint32_t*)r,
                                                                               (const uint32_t*)okp, ad, ad_off, valid, zinv, proof, blinding);
  LAUNCHED_AS(ctx, "pedersen_prove_finish");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_pedersen_prove_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output,
                                                 const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_proof, uint8_t* out_blinding) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !input || !output || !out_proof || !out_blinding) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_pr, *d_bl;
  HostIn in[3] = {{BUF_IN0, sk, 32, true, nullptr}, {BUF_IN1, input, 64, false, nullptr}, {BUF_IN2, output, 64, false, nullptr}};
  Pieces pc;   // 288 B/item of results: worth VRFS_HOST_PIECES pieces (measured 2^20: e2e 19.4 -> 20.8 M/s, kernels 21.8 -> 20.9 M/s)
  ST(stage_in_pieces(ctx, n, in, 3, &pc, VRFS_HOST_PIECES));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n * 256, &d_pr)); ST(stage_out(ctx, BUF_OUT1, n * 32, &d_bl));
  mark_secret(ctx, BUF_OUT1, n * 32);
  const HostOut out[2] = {{out_proof, d_pr, 256}, {out_blinding, d_bl, 32}};
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
      return pedersen_prove_dev<S>(ctx, m, in[0].dev + o * 32, in[1].dev + o * 64, in[2].dev + o * 64, d_ad, d_off ? d_off + o : nullptr, d_pr + o * 256, d_bl + o * 32); }));
    ST(pieces_copy_out(ctx, pc, k, out, 2));
  }
  return finish_call(ctx);
}
template <class S>
static vrfs_status pedersen_verify_dev(vrfs_ctx* ctx, size_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof, const uint8_t* ad,
                                       const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status = nullptr) {
  typedef typename S::C C;
  void *c = nullptr, *t1 = nullptr, *t2 = nullptr;
  uint8_t* valid = nullptr;
  ST(need_tables<S>(ctx));
  ST(ensure(ctx, BUF_W0, n * 32, &c)); ST(ensure(ctx, BUF_W1, n * 96, &t1)); ST(ensure(ctx, BUF_W2, n * 96, &t2));
  ST(fresh_valid(ctx, n, &valid));
  k_pedersen_verify_prep<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, input, output, proof, ad, ad_off, (uint8_t*)c, valid);
  LAUNCHED_AS(ctx, "pedersen_verify_prep");
  LincombArgs A = {};
  A.n = (uint32_t)n; A.valid = valid;
  // T1 = s*I - c*O
  const uint32_t cbits = S::CLEN < 32 ? 8u * S::CLEN : 0u;
  A.var[0] = {input, 64, proof + 192, 256, 0, 0}; A.var[1] = {output, 64, (const uint8_t*)c, 32, 1, cbits}; A.out_xyz = (uint32_t*)t1;
  ST((launch_lincomb<C, 2, 0>(ctx, A)));
  // T2 = s*G + sb*B - c*Yb
  A.var[0] = {proof, 256, (const uint8_t*)c, 32, 1, cbits};
  A.fix[0] = {proof + 192, 256, 0, fixtab<S>(ctx, 0)}; A.fix[1] = {proof + 224, 256, 0, fixtab<S>(ctx, 1)}; A.out_xyz = (uint32_t*)t2;
  ST((launch_lincomb<C, 1, 2>(ctx, A)));
  k_pedersen_verify_finish<C><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, proof, (const uint32_t*)t1, (const uint32_t*)t2, valid, out_ok, out_status);
  LAUNCHED_AS(ctx, "pedersen_verify_finish");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_pedersen_verify_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof,
                                                  const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!input || !output || !proof || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_ok, *d_st = nullptr;
  HostIn in[3] = {{BUF_IN0, input, 64, false, nullptr}, {BUF_IN1, output, 64, false, nullptr}, {BUF_IN2, proof, 256, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 3, &pc, 2));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
      return pedersen_verify_dev<S>(ctx, m, in[0].dev + o * 64, in[1].dev + o * 64, in[2].dev + o * 256, d_ad, d_off ? d_off + o : nullptr, d_ok + o, d_st ? d_st + o : nullptr); }));
  }
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}

// =================================================================================================
// wire formats (SURVEY 8f-1): serialised keys / signatures in, verdicts out
// =================================================================================================
// Public / Output deserialisation: codec decode + on-curve + prime-order subgroup.  One thread per encoded point; `enc_b`
// (stride_b) is an optional second array processed by threads n..2n-1 (the verify path decodes keys and gammas together).
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_decode_checked(uint32_t n, const uint8_t* enc_a, uint32_t stride_a, uint8_t* out_a,
                                                                                     const uint8_t* enc_b, uint32_t stride_b, uint8_t* out_b, uint8_t* flags) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (enc_b ? 2 * n : n)) return;
  const bool second = t >= n;
  const uint32_t i = second ? t - n : t;
  const uint8_t* e = second ? enc_b + (size_t)stride_b * i : enc_a + (size_t)stride_a * i;
  uint8_t tmp[S::ENC_LEN];
  for (int j = 0; j < S::ENC_LEN; j++) tmp[j] = e[j];
  flags[t] = (uint8_t)wire_decode_point_checked<S>((second ? out_b : out_a) + (size_t)64 * i, tmp);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_subgroup_check(uint32_t n, const uint8_t* pts, uint8_t* out_ok) {
  ITEM_INDEX(n);
  typedef typename S::C C;
  typename C::F x, y;
  bool inf = false;
  bool ok = load_affine<C>(x, y, &inf, pts + (size_t)64 * i);
  out_ok[i] = (uint8_t)(ok && (inf || SubgroupCheck<C>::run(x, y)));
}
// ietf::Proof deserialisation + merge of the two point flags
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_wire_parse_proof(uint32_t n, const uint8_t* sig, const uint8_t* flags2, uint8_t* c, uint8_t* s, uint8_t* valid) {
  ITEM_INDEX(n);
  constexpr int SL = S::ENC_LEN + S::CLEN + 32;
  bool ok = wire_parse_proof<S>(c + (size_t)32 * i, s + (size_t)32 * i, sig + (size_t)SL * i + S::ENC_LEN);
  valid[i] = (uint8_t)(ok && flags2[i] && flags2[n + i]);
}
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_wire_pack_sig(uint32_t n, const uint8_t* output, const uint8_t* c, const uint8_t* s, const uint8_t* ok, uint8_t* sig) {
  ITEM_INDEX(n);
  constexpr int SL = S::ENC_LEN + S::CLEN + 32;
  uint8_t* o = sig + (size_t)SL * i;
  if (!ok[i]) { for (int j = 0; j < SL; j++) o[j] = 0; return; }
  uint8_t tmp[SL];
  wire_pack_signature<S>(tmp, output + (size_t)64 * i, c + (size_t)32 * i, s + (size_t)32 * i);
  for (int j = 0; j < SL; j++) o[j] = tmp[j];
}
// out_ok &= a & b; rejected items get a zero hash; a failed deserialisation (a or b clear) is Error::InvalidData
__global__ void k_merge_flags(uint32_t n, const uint8_t* a, const uint8_t* b, uint8_t* out_ok, uint8_t* hash, uint32_t hlen, uint8_t* status) {
  ITEM_INDEX(n);
  const uint8_t wellformed = a[i] & (b ? b[i] : 1);
  uint8_t ok = out_ok[i] & wellformed;
  out_ok[i] = ok;
  if (status) status[i] = (uint8_t)(ok ? ITEM_OK : !wellformed ? ITEM_INVALID_DATA : status[i] == ITEM_OK ? ITEM_VERIFICATION_FAILURE : status[i]);
  if (hash && !ok) for (uint32_t j = 0; j < hlen; j++) hash[(size_t)hlen * i + j] = 0;
}
// signature against a prepared key named by index (vrfs_ietf_verify_prepared_wire_batch), in place of k_decode_checked (key and
// Output), k_wire_parse_proof and k_gather_keys: item i's key row (zeros for an index out of range), its Output decoded with the
// subgroup check, c and s parsed.  valid[i] = the index names a valid key (what k_gather_keys leaves); wellformed[i] = that and
// both deserialisations succeeded (k_merge_flags' `a`, which the wire call takes from k_wire_parse_proof)
template <class S> __global__ void __launch_bounds__(ITEM_THREADS) k_wire_prepared_unpack(uint32_t n, const uint32_t* key_index, uint32_t n_keys, const uint8_t* rows,
                                                                                           const uint8_t* key_ok, const uint8_t* sig, uint8_t* out_rows, uint8_t* output,
                                                                                           uint8_t* c, uint8_t* s, uint8_t* valid, uint8_t* wellformed) {
  ITEM_INDEX(n);
  constexpr uint32_t SL = S::ENC_LEN + S::CLEN + 32;
  const uint8_t* e = sig + (size_t)SL * i;
  uint8_t tmp[S::ENC_LEN];
  for (int j = 0; j < S::ENC_LEN; j++) tmp[j] = e[j];
  const bool out_ok = wire_decode_point_checked<S>(output + (size_t)64 * i, tmp);
  const bool parsed = wire_parse_proof<S>(c + (size_t)32 * i, s + (size_t)32 * i, e + S::ENC_LEN);
  const uint32_t k = key_index[i];                               // after the decode: nothing of the key is live across it
  const bool key = k < n_keys && key_ok[k];
  uint4 r[4] = {};
  if (k < n_keys) copy_words16(&r, reinterpret_cast<const uint4(*)[4]>(rows) + k);
  copy_words16(reinterpret_cast<uint4(*)[4]>(out_rows) + i, &r);
  valid[i] = (uint8_t)key;
  wellformed[i] = (uint8_t)(key && out_ok && parsed);
}

extern "C" int vrfs_suite_ietf_signature_len(vrfs_suite s) { return vrfs_suite_point_enc_len(s) + vrfs_suite_challenge_len(s) + 32; }

template <class S> static vrfs_status decode_checked_launch(vrfs_ctx* ctx, size_t n, const uint8_t* a, uint32_t sa, uint8_t* oa, const uint8_t* b, uint32_t sb, uint8_t* ob, uint8_t* flags) {
  const size_t threads = b ? 2 * n : n;
  k_decode_checked<S><<<item_blocks(threads), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, a, sa, oa, b, sb, ob, flags);
  LAUNCHED_AS(ctx, "decode_checked");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_point_decode_checked_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* enc, uint8_t* out_pts, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!enc || !out_pts || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint32_t el = (uint32_t)vrfs_suite_point_enc_len(suite);
  const uint8_t* d_e; uint8_t *d_p, *d_ok;
  ST(stage_in(ctx, BUF_X0, enc, n * el, &d_e)); ST(stage_out(ctx, BUF_OUT0, n * 64, &d_p)); ST(stage_out(ctx, BUF_OUT1, n, &d_ok));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return decode_checked_launch<S>(ctx, n, d_e, el, d_p, nullptr, 0, nullptr, d_ok); }));
  ST(copy_out(ctx, out_pts, d_p, n * 64)); ST(copy_out(ctx, out_ok, d_ok, n));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_subgroup_check_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pts, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!pts || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const uint8_t* d_p; uint8_t* d_ok;
  ST(stage_in(ctx, BUF_IN0, pts, n * 64, &d_p)); ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; k_subgroup_check<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, d_p, d_ok); return VRFS_OK; }));
  LAUNCHED_AS(ctx, "subgroup_check");
  ST(copy_out(ctx, out_ok, d_ok, n));
  return finish_call(ctx);
}

// Secret -> signature: Input::new(data), Secret::output, ietf::Prover::prove, serialise
template <class S> static vrfs_status ietf_sign_wire_dev(vrfs_ctx* ctx, size_t n, const uint8_t* sk, const uint8_t* data, const uint64_t* data_off,
                                                         const uint8_t* ad, const uint64_t* ad_off, uint8_t* input, uint8_t* output, uint8_t* c, uint8_t* s,
                                                         uint8_t* h2c_ok, uint8_t* sig) {
  ST(data_to_point_dev<S>(ctx, n, data, data_off, input, h2c_ok));
  ST(output_dev<S>(ctx, n, sk, input, output));
  ST(ietf_prove_dev<S>(ctx, n, sk, input, output, ad, ad_off, c, s));
  k_wire_pack_sig<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, output, c, s, h2c_ok, sig);
  LAUNCHED_AS(ctx, "wire_pack_sig");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ietf_sign_wire_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* data, const uint64_t* data_off,
                                                 const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_sig, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !data_off || !out_sig) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const size_t sl = (size_t)vrfs_suite_ietf_signature_len(suite);
  const uint8_t *d_sk, *d_ad, *d_data; const uint64_t *d_off, *d_doff;
  uint8_t *d_in, *d_out, *d_c, *d_s, *d_ok, *d_sig;
  ST(stage_secret(ctx, BUF_IN0, sk, n * 32, &d_sk));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_var(ctx, BUF_X2, BUF_X3, n, data, data_off, &d_data, &d_doff));
  ST(stage_out(ctx, BUF_IN1, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN2, n * 64, &d_out)); ST(stage_out(ctx, BUF_IN3, n * 32, &d_c)); ST(stage_out(ctx, BUF_IN4, n * 32, &d_s));
  ST(stage_out(ctx, BUF_X4, n, &d_ok)); ST(stage_out(ctx, BUF_X1, n * sl, &d_sig));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return ietf_sign_wire_dev<S>(ctx, n, d_sk, d_data, d_doff, d_ad, d_off, d_in, d_out, d_c, d_s, d_ok, d_sig); }));
  ST(copy_out(ctx, out_sig, d_sig, n * sl));
  if (out_ok) ST(copy_out(ctx, out_ok, d_ok, n));
  return finish_call(ctx);
}

// serialised Public + data + signature -> verdict (+ Output::hash of accepted items)
template <class S> static vrfs_status ietf_verify_wire_dev(vrfs_ctx* ctx, size_t n, const uint8_t* pk_enc, const uint8_t* data, const uint64_t* data_off, const uint8_t* sig,
                                                           const uint8_t* ad, const uint64_t* ad_off, uint8_t* pk, uint8_t* input, uint8_t* output, uint8_t* c, uint8_t* s,
                                                           uint8_t* flags /*4n*/, uint8_t* out_ok, uint8_t* out_hash, uint8_t* out_status) {
  constexpr uint32_t SL = S::ENC_LEN + S::CLEN + 32;
  ST((decode_checked_launch<S>(ctx, n, pk_enc, S::ENC_LEN, pk, sig, SL, output, flags)));
  k_wire_parse_proof<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sig, flags, c, s, flags + 2 * n);
  LAUNCHED_AS(ctx, "wire_parse_proof");
  ST(data_to_point_dev<S>(ctx, n, data, data_off, input, flags + 3 * n));
  ST(ietf_verify_dev<S>(ctx, n, pk, input, output, c, s, ad, ad_off, out_ok, out_status));
  if (out_hash) {
    k_point_to_hash<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, output, out_hash);
    LAUNCHED_AS(ctx, "point_to_hash");
  }
  k_merge_flags<<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, flags + 2 * n, flags + 3 * n, out_ok, out_hash, (uint32_t)S::HLEN, out_status);
  LAUNCHED_AS(ctx, "merge_flags");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ietf_verify_wire_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* pk_enc, const uint8_t* data, const uint64_t* data_off,
                                                   const uint8_t* sig, const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_hash, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!pk_enc || !data_off || !sig || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const size_t sl = (size_t)vrfs_suite_ietf_signature_len(suite), el = (size_t)vrfs_suite_point_enc_len(suite), hl = (size_t)vrfs_suite_hash_len(suite);
  const uint8_t *d_ad, *d_data; const uint64_t *d_off, *d_doff;
  uint8_t *d_pk, *d_in, *d_out, *d_c, *d_s, *d_flags, *d_ok, *d_hash = nullptr, *d_st = nullptr;
  // keys and signatures on the copy stream, enqueued first: the host-side checks of the offset arrays below run while they
  // travel; the variable-length data and ad go on the main stream.  ONE piece: with [one wave, rest] the decode and
  // hash-to-curve kernels of the small first piece run below their full-batch rate and the call as a whole was 1.3 % slower
  // (2^20 Bandersnatch items, 9.07 -> 8.96 M/s).
  HostIn in[2] = {{BUF_X0, pk_enc, el, false, nullptr}, {BUF_X1, sig, sl, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 2, &pc, 1));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_var(ctx, BUF_X2, BUF_X3, n, data, data_off, &d_data, &d_doff));
  ST(stage_out(ctx, BUF_IN0, n * 64, &d_pk)); ST(stage_out(ctx, BUF_IN1, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN2, n * 64, &d_out));
  ST(stage_out(ctx, BUF_IN3, n * 32, &d_c)); ST(stage_out(ctx, BUF_IN4, n * 32, &d_s)); ST(stage_out(ctx, BUF_X4, 4 * n, &d_flags));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_hash) ST(stage_out(ctx, BUF_OUT1, n * hl, &d_hash));
  if (out_status) ST(stage_out(ctx, BUF_X5, n, &d_st));
  HostOut out[3] = {{out_ok, d_ok, 1}, {nullptr, nullptr, 0}, {nullptr, nullptr, 0}};
  int nout = 1;
  if (out_hash) out[nout++] = {out_hash, d_hash, hl};
  if (out_status) out[nout++] = {out_status, d_st, 1};
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_verify_wire_dev<S>(ctx, m, in[0].dev + o * el, d_data, d_doff + o, in[1].dev + o * sl, d_ad, d_off ? d_off + o : nullptr, d_pk + o * 64, d_in + o * 64,
                                     d_out + o * 64, d_c + o * 32, d_s + o * 32, d_flags + o * 4, d_ok + o, d_hash ? d_hash + o * hl : nullptr, d_st ? d_st + o : nullptr); }));
    ST(pieces_copy_out(ctx, pc, k, out, nout));
  }
  return finish_call(ctx);
}

// ---- pedersen on the wire.  Two layouts share the kernels below (NP = encoded points per item):
//   NP = 4  signature: point_encode(Output) || point_encode(pk_com) || point_encode(r) || point_encode(ok) || s || sb
//           (an `Output` followed by `pedersen::Proof`'s CanonicalSerialize, A.10; Bandersnatch 192 B)
//   NP = 3  the typed `pedersen::Proof` alone: pk_com || r || ok || s || sb (Bandersnatch 160 B, SURVEY 8b)
// one thread per encoded point: with NP = 4 point 0 goes to output_aff[item]; the proof's points go to the 256-byte ABI proof
template <class S, int NP> __global__ void __launch_bounds__(ITEM_THREADS) k_ped_wire_points(uint32_t n, const uint8_t* sig, uint8_t* output, uint8_t* proof256, uint8_t* flags) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= NP * n) return;
  constexpr uint32_t SL = NP * S::ENC_LEN + 64;
  const uint32_t j = t / n, i = t % n;
  const uint8_t* e = sig + (size_t)SL * i + (size_t)S::ENC_LEN * j;
  uint8_t tmp[S::ENC_LEN];
  for (int k = 0; k < S::ENC_LEN; k++) tmp[k] = e[k];
  const uint32_t slot = NP == 4 ? j - 1 : j;
  uint8_t* dst = (NP == 4 && j == 0) ? output + (size_t)64 * i : proof256 + (size_t)256 * i + 64 * slot;
  flags[t] = (uint8_t)wire_decode_point_checked<S>(dst, tmp);
}
template <class S, int NP> __global__ void __launch_bounds__(ITEM_THREADS) k_ped_wire_scalars(uint32_t n, const uint8_t* sig, const uint8_t* flagsNP, uint8_t* proof256, uint8_t* valid) {
  ITEM_INDEX(n);
  constexpr uint32_t SL = NP * S::ENC_LEN + 64;
  const uint8_t* p = sig + (size_t)SL * i + NP * S::ENC_LEN;
  uint8_t* o = proof256 + (size_t)256 * i + 192;
  bool ok = true;
  for (int h = 0; h < 2; h++) {
    for (int j = 0; j < 32; j++) o[32 * h + j] = S::SEC1 ? p[32 * h + 31 - j] : p[32 * h + j];
    uint32_t raw[8];
    load_le<8>(raw, o + 32 * h);
    ok &= is_canonical<typename S::C::Fr>(raw);
  }
  for (int j = 0; j < NP; j++) ok &= flagsNP[(size_t)j * n + i] != 0;
  valid[i] = (uint8_t)ok;
}
template <class S, int NP> __global__ void __launch_bounds__(ITEM_THREADS) k_ped_wire_pack(uint32_t n, const uint8_t* output, const uint8_t* proof256, const uint8_t* ok, uint8_t* sig) {
  ITEM_INDEX(n);
  constexpr uint32_t SL = NP * S::ENC_LEN + 64;
  uint8_t* o = sig + (size_t)SL * i;
  if (ok && !ok[i]) { for (uint32_t j = 0; j < SL; j++) o[j] = 0; return; }
  const uint8_t* pr = proof256 + (size_t)256 * i;
  uint8_t tmp[SL];
  if (NP == 4) encode_point_bytes<S>(tmp, output + (size_t)64 * i);
  for (int j = 0; j < 3; j++) encode_point_bytes<S>(tmp + S::ENC_LEN * (j + NP - 3), pr + 64 * j);
  for (int h = 0; h < 2; h++) for (int j = 0; j < 32; j++) tmp[NP * S::ENC_LEN + 32 * h + j] = S::SEC1 ? pr[192 + 32 * h + 31 - j] : pr[192 + 32 * h + j];
  for (uint32_t j = 0; j < SL; j++) o[j] = tmp[j];
}
extern "C" int vrfs_suite_pedersen_signature_len(vrfs_suite s) { return 4 * vrfs_suite_point_enc_len(s) + 64; }
extern "C" int vrfs_suite_pedersen_proof_len(vrfs_suite s) { return 3 * vrfs_suite_point_enc_len(s) + 64; }

template <class S> static vrfs_status pedersen_sign_wire_dev(vrfs_ctx* ctx, size_t n, const uint8_t* sk, const uint8_t* data, const uint64_t* data_off, const uint8_t* ad,
                                                             const uint64_t* ad_off, uint8_t* input, uint8_t* output, uint8_t* proof256, uint8_t* blinding, uint8_t* h2c_ok, uint8_t* sig) {
  ST(data_to_point_dev<S>(ctx, n, data, data_off, input, h2c_ok));
  ST(output_dev<S>(ctx, n, sk, input, output));
  ST(pedersen_prove_dev<S>(ctx, n, sk, input, output, ad, ad_off, proof256, blinding));
  k_ped_wire_pack<S, 4><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, output, proof256, h2c_ok, sig);
  LAUNCHED_AS(ctx, "ped_wire_pack");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_pedersen_sign_wire_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* data, const uint64_t* data_off,
                                                     const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_sig, uint8_t* out_blinding, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !data_off || !out_sig || !out_blinding) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const size_t sl = (size_t)vrfs_suite_pedersen_signature_len(suite);
  const uint8_t *d_sk, *d_ad, *d_data; const uint64_t *d_off, *d_doff;
  uint8_t *d_in, *d_out, *d_pr, *d_bl, *d_ok, *d_sig;
  ST(stage_secret(ctx, BUF_IN0, sk, n * 32, &d_sk));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_var(ctx, BUF_X2, BUF_X3, n, data, data_off, &d_data, &d_doff));
  ST(stage_out(ctx, BUF_IN1, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN2, n * 64, &d_out)); ST(stage_out(ctx, BUF_OUT0, n * 256, &d_pr)); ST(stage_out(ctx, BUF_OUT1, n * 32, &d_bl));
  mark_secret(ctx, BUF_OUT1, n * 32);
  ST(stage_out(ctx, BUF_X4, n, &d_ok)); ST(stage_out(ctx, BUF_X1, n * sl, &d_sig));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return pedersen_sign_wire_dev<S>(ctx, n, d_sk, d_data, d_doff, d_ad, d_off, d_in, d_out, d_pr, d_bl, d_ok, d_sig); }));
  ST(copy_out(ctx, out_sig, d_sig, n * sl)); ST(copy_out(ctx, out_blinding, d_bl, n * 32));
  if (out_ok) ST(copy_out(ctx, out_ok, d_ok, n));
  return finish_call(ctx);
}
// deserialise NP encoded points + 2 scalars per item, then pedersen::Verifier::verify.  NP = 4: input = Input::new(data) here
// (h2c flags in flags[(NP+1)n ..]); NP = 3: input and output are the caller's typed values.
template <class S, int NP> static vrfs_status pedersen_wire_decode_dev(vrfs_ctx* ctx, size_t n, const uint8_t* data, const uint64_t* data_off, const uint8_t* sig,
                                                                       uint8_t* input, uint8_t* output, uint8_t* proof256, uint8_t* flags /*(NP+2)n*/) {
  k_ped_wire_points<S, NP><<<item_blocks(NP * n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sig, output, proof256, flags);
  LAUNCHED_AS(ctx, "decode_checked");
  k_ped_wire_scalars<S, NP><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, sig, flags, proof256, flags + NP * n);
  LAUNCHED_AS(ctx, "ped_wire_scalars");
  if (NP == 4) ST(data_to_point_dev<S>(ctx, n, data, data_off, input, flags + (NP + 1) * n));
  return VRFS_OK;
}
template <class S, int NP> static vrfs_status pedersen_wire_verdicts_dev(vrfs_ctx* ctx, size_t n, const uint8_t* ad, const uint64_t* ad_off, const uint8_t* input,
                                                                         const uint8_t* output, const uint8_t* proof256, const uint8_t* flags, uint8_t* out_ok, uint8_t* out_status) {
  ST(pedersen_verify_dev<S>(ctx, n, input, output, proof256, ad, ad_off, out_ok, out_status));
  k_merge_flags<<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, flags + NP * n, NP == 4 ? flags + (NP + 1) * n : nullptr, out_ok, nullptr, 0u, out_status);
  LAUNCHED_AS(ctx, "merge_flags");
  return VRFS_OK;
}
template <class S, int NP> static vrfs_status pedersen_verify_wire_dev(vrfs_ctx* ctx, size_t n, const uint8_t* data, const uint64_t* data_off, const uint8_t* sig, const uint8_t* ad,
                                                                       const uint64_t* ad_off, uint8_t* input, uint8_t* output, uint8_t* proof256, uint8_t* flags /*(NP+2)n*/,
                                                                       uint8_t* out_ok, uint8_t* out_status) {
  ST((pedersen_wire_decode_dev<S, NP>(ctx, n, data, data_off, sig, input, output, proof256, flags)));
  return pedersen_wire_verdicts_dev<S, NP>(ctx, n, ad, ad_off, input, output, proof256, flags, out_ok, out_status);
}
extern "C" vrfs_status vrfs_pedersen_verify_wire_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* data, const uint64_t* data_off, const uint8_t* sig,
                                                       const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!data_off || !sig || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const size_t sl = (size_t)vrfs_suite_pedersen_signature_len(suite);
  const uint8_t *d_sig, *d_ad, *d_data; const uint64_t *d_off, *d_doff;
  uint8_t *d_in, *d_out, *d_pr, *d_flags, *d_ok, *d_st = nullptr;
  ST(stage_in(ctx, BUF_X1, sig, n * sl, &d_sig));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_var(ctx, BUF_X2, BUF_X3, n, data, data_off, &d_data, &d_doff));
  ST(stage_out(ctx, BUF_IN0, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN1, n * 64, &d_out)); ST(stage_out(ctx, BUF_IN2, n * 256, &d_pr));
  ST(stage_out(ctx, BUF_X4, 6 * n, &d_flags)); ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return (pedersen_verify_wire_dev<S, 4>(ctx, n, d_data, d_doff, d_sig, d_ad, d_off, d_in, d_out, d_pr, d_flags, d_ok, d_st)); }));
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}

// ---- the typed pedersen::Proof in its serialised form (3 encoded points + 2 scalars: 160 B for Bandersnatch; SURVEY 8b) ----
template <class S> static vrfs_status pedersen_prove_compressed_dev(vrfs_ctx* ctx, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output, const uint8_t* ad,
                                                                    const uint64_t* ad_off, uint8_t* proof256, uint8_t* blinding, uint8_t* out) {
  ST(pedersen_prove_dev<S>(ctx, n, sk, input, output, ad, ad_off, proof256, blinding));
  k_ped_wire_pack<S, 3><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, nullptr, proof256, nullptr, out);
  LAUNCHED_AS(ctx, "ped_wire_pack");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_pedersen_prove_compressed_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output,
                                                            const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_proof, uint8_t* out_blinding) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!sk || !input || !output || !out_proof || !out_blinding) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const size_t pl = (size_t)vrfs_suite_pedersen_proof_len(suite);
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_pr, *d_bl, *d_enc;
  HostIn in[3] = {{BUF_IN0, sk, 32, true, nullptr}, {BUF_IN1, input, 64, false, nullptr}, {BUF_IN2, output, 64, false, nullptr}};
  Pieces pc;   // in pieces like vrfs_pedersen_prove_batch: 192 B/item of results (Bandersnatch) return beside the next piece's kernels
  ST(stage_in_pieces(ctx, n, in, 3, &pc, VRFS_HOST_PIECES));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n * 256, &d_pr)); ST(stage_out(ctx, BUF_OUT1, n * 32, &d_bl)); ST(stage_out(ctx, BUF_X1, n * pl, &d_enc));
  mark_secret(ctx, BUF_OUT1, n * 32);
  const HostOut out[2] = {{out_proof, d_enc, pl}, {out_blinding, d_bl, 32}};
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
      return pedersen_prove_compressed_dev<S>(ctx, m, in[0].dev + o * 32, in[1].dev + o * 64, in[2].dev + o * 64, d_ad, d_off ? d_off + o : nullptr,
                                              d_pr + o * 256, d_bl + o * 32, d_enc + o * pl); }));
    ST(pieces_copy_out(ctx, pc, k, out, 2));
  }
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_pedersen_verify_compressed_batch(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof,
                                                             const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n == 0) return VRFS_OK;
  if (!input || !output || !proof || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, suite, n));
  const size_t pl = (size_t)vrfs_suite_pedersen_proof_len(suite);
  const uint8_t *d_enc, *d_ad, *d_in, *d_out; const uint64_t* d_off;
  uint8_t *d_pr, *d_flags, *d_ok, *d_st = nullptr;
  ST(stage_in(ctx, BUF_X1, proof, n * pl, &d_enc));
  ST(stage_in(ctx, BUF_IN0, input, n * 64, &d_in)); ST(stage_in(ctx, BUF_IN1, output, n * 64, &d_out));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_IN2, n * 256, &d_pr)); ST(stage_out(ctx, BUF_X4, 5 * n, &d_flags)); ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  uint8_t *m_in = const_cast<uint8_t*>(d_in), *m_out = const_cast<uint8_t*>(d_out);
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return (pedersen_verify_wire_dev<S, 3>(ctx, n, nullptr, nullptr, d_enc, d_ad, d_off, m_in, m_out, d_pr, d_flags, d_ok, d_st)); }));
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}

// =================================================================================================
// Pedersen batch verification by one random linear combination (Bandersnatch only; DESIGN §4 "Pedersen batch verification")
// =================================================================================================
//   E_i = Ok_i + c_i O_i - s_i I_i,   F_i = R_i + c_i Yb_i - s_i G - sb_i B      (both 0 for a valid proof)
// The batch is accepted iff  sum_i rho_i E_i + sigma_i F_i = 0: one MSM (csrc/te_msm.cuh) over the 5n + 2 bases
// [Ok, O, I, R, Yb of every item | G | B] with the scalars [rho, rho c, -rho s, sigma, sigma c | -sum sigma s | -sum sigma sb].
// With every point in the prime-order subgroup a non-zero E_j or F_j survives all but one value of its coefficient (false accept
// <= 2^-127); a 2-torsion component would vanish under every even one.  So the five points of every item are subgroup-checked
// (typed inputs) or come from the checked wire decoder (`SUBGROUP` = false), and any failure sets the batch's `bad` flag.
#define PED_BATCH_NP 5
template <class S, bool SUBGROUP>
__global__ void __launch_bounds__(ITEM_THREADS) k_pedersen_batch_prep(uint32_t n, uint32_t first, const uint8_t* input, const uint8_t* output, const uint8_t* proof,
                                                                      const uint8_t* ad, const uint64_t* ad_off, const uint8_t* valid0, const uint8_t* valid1,
                                                                      const uint8_t* seed, BandAff* bases, uint8_t* scal, uint32_t* prod, uint32_t* bad) {
  ITEM_INDEX(n);
  typedef typename S::C C;
  typedef typename C::Fr R;
  typedef Fp<R> Fr;
  VAR_SLICE(ad, ad_off, i, a, alen);
  const uint8_t* pr = proof + (size_t)256 * i;
  const size_t g = (size_t)first + i;                              // index of the item in the whole batch
  uint8_t c32[32];
  bool ok = pedersen_verify_prep_item<S>(c32, input + (size_t)64 * i, output + (size_t)64 * i, pr, a, alen);
  if (valid0) ok &= valid0[i] != 0;
  if (valid1) ok &= valid1[i] != 0;
  const uint8_t* pts[PED_BATCH_NP] = {pr + 128, output + (size_t)64 * i, input + (size_t)64 * i, pr + 64, pr};   // Ok, O, I, R, Yb
  for (int j = 0; j < PED_BATCH_NP; j++) {
    uint32_t rx[8], ry[8];
    load_le<8>(rx, pts[j]); load_le<8>(ry, pts[j] + 32);
    bool pok = is_canonical<typename C::Fq>(rx) & is_canonical<typename C::Fq>(ry);
    const typename C::F x = to_mont<typename C::Fq>(rx), y = to_mont<typename C::Fq>(ry);
    pok &= Grp<C>::on_curve(x, y);
    if (SUBGROUP && pok) pok = SubgroupCheck<C>::run(x, y);
    ok &= pok;
    BandAff e; band_aff_from_xy(e, x, y);
    copy_words16(&bases[PED_BATCH_NP * g + j], &e);
  }
  // (rho || sigma) = the first 32 bytes of SHA-512("vrfs-b200/pedersen-batch/v1" || seed || LE64(g) || c), two 16-byte
  // little-endian halves with bit 127 cleared
  constexpr char dom[] = "vrfs-b200/pedersen-batch/v1";
  Sha512 h; h.init();
  for (int k = 0; k + 1 < (int)sizeof(dom); k++) h.put((uint8_t)dom[k]);
  h.update(seed, 32);
  for (int k = 0; k < 8; k++) h.put((uint8_t)((uint64_t)g >> (8 * k)));
  h.update(c32, 32);
  uint8_t dig[64]; h.final(dig);
  uint32_t raw[8];
  Fr coef[2];
  for (int half = 0; half < 2; half++) {
    for (int k = 4; k < 8; k++) raw[k] = 0;
    load_le<4>(raw, dig + 16 * half);
    raw[3] &= 0x7fffffffu;
    coef[half] = to_mont<R>(raw);
  }
  load_le<8>(raw, c32); const Fr c = to_mont<R>(raw);
  load_le<8>(raw, pr + 192); const Fr s = to_mont<R>(raw);           // reduced mod r on load, as the per-item verifier does
  load_le<8>(raw, pr + 224); const Fr sb = to_mont<R>(raw);
  const Fr k5[PED_BATCH_NP] = {coef[0], coef[0] * c, neg(coef[0] * s), coef[1], coef[1] * c};
  for (int j = 0; j < PED_BATCH_NP; j++) { from_mont<R>(raw, k5[j]); store_le<8>(scal + (size_t)32 * (PED_BATCH_NP * g + j), raw); }
  const Fr ss = coef[1] * s, ssb = coef[1] * sb;
  for (int w = 0; w < 8; w++) { prod[(size_t)16 * g + w] = ss.v[w]; prod[(size_t)16 * g + 8 + w] = ssb.v[w]; }
  if (!ok) *bad = 1u;
}
// sum_i sigma_i s_i and sum_i sigma_i sb_i (Montgomery words, 16 per item): every block adds a strided slice into partial[block];
// launched again as one block over those partials (`last`), which writes the scalars of G and B, -sum sigma s and -sum sigma sb mod r,
// and their affine-cached records behind the nitems items
__global__ void __launch_bounds__(256) k_pedersen_batch_sum(uint32_t n, const uint32_t* prod, uint32_t* partial, int last, uint32_t nitems, BandAff* bases, uint8_t* scal) {
  typedef Fp<BandFr> Fr;
  __shared__ uint32_t sh[256][16];
  Fr a = Fr::zero(), b = Fr::zero();
  for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
    Fr p, q;
    for (int j = 0; j < 8; j++) { p.v[j] = prod[(size_t)16 * i + j]; q.v[j] = prod[(size_t)16 * i + 8 + j]; }
    a = a + p; b = b + q;
  }
  for (int j = 0; j < 8; j++) { sh[threadIdx.x][j] = a.v[j]; sh[threadIdx.x][8 + j] = b.v[j]; }
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) {
      Fr p, q;
      for (int j = 0; j < 8; j++) { p.v[j] = sh[threadIdx.x + s][j]; q.v[j] = sh[threadIdx.x + s][8 + j]; }
      a = a + p; b = b + q;
      for (int j = 0; j < 8; j++) { sh[threadIdx.x][j] = a.v[j]; sh[threadIdx.x][8 + j] = b.v[j]; }
    }
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  if (!last) { for (int j = 0; j < 8; j++) { partial[16 * blockIdx.x + j] = a.v[j]; partial[16 * blockIdx.x + 8 + j] = b.v[j]; } return; }
  uint32_t out[8];
  from_mont<BandFr>(out, neg(a)); store_le<8>(scal + (size_t)32 * (PED_BATCH_NP * (size_t)nitems), out);
  from_mont<BandFr>(out, neg(b)); store_le<8>(scal + (size_t)32 * (PED_BATCH_NP * (size_t)nitems + 1), out);
  BandAff e;
  band_aff_from_xy(e, BandCurve::gx(), BandCurve::gy()); copy_words16(&bases[PED_BATCH_NP * (size_t)nitems], &e);
  band_aff_from_xy(e, BandCurve::bx(), BandCurve::by()); copy_words16(&bases[PED_BATCH_NP * (size_t)nitems + 1], &e);
}
#define PED_BATCH_SUM_BLOCKS 1024

// Device state of one batch verification, in slots of its own (BUF_PB*): a rejected batch runs the per-item verifier next, which
// reuses the work buffers W*, VALID and SLAB but must find the staged inputs (IN*, AD, OFF, X*) intact.
struct PedBatch { BandAff* bases; uint8_t* scal; uint32_t* prod; uint32_t* partial; uint32_t* bad; uint8_t* verdict; uint8_t* seed; };
static vrfs_status ped_batch_begin(vrfs_ctx* ctx, vrfs_suite suite, size_t n) {
  ST(begin_call(ctx, suite, n));
  if (suite != VRFS_BANDERSNATCH_ELL2)
    return fail(ctx, VRFS_UNSUPPORTED, "batch verification by random linear combination needs points of prime order, and only Bandersnatch has a cheap subgroup test "
                                       "(the cofactor-8 curves need a full [r]P per point; short-Weierstrass curves have no bucket MSM here): use vrfs_pedersen_verify_batch");
  if (n > (1u << 24)) return fail(ctx, VRFS_BAD_ARG, "more than 2^24 proofs per batch verification are not supported");
  return VRFS_OK;
}
static vrfs_status ped_batch_alloc(vrfs_ctx* ctx, size_t n, const uint8_t* seed, PedBatch* B) {
  const size_t nbases = PED_BATCH_NP * n + 2;
  void *b = nullptr, *s = nullptr, *m = nullptr;
  ST(ensure(ctx, BUF_PB0, nbases * sizeof(BandAff), &b));
  ST(ensure(ctx, BUF_PB1, nbases * 32, &s));
  ST(ensure(ctx, BUF_PB2, 256 + (n + PED_BATCH_SUM_BLOCKS) * 64, &m));   // seed (32 B) | bad flag | verdict | ... | prod (n x 16 words) | partial sums
  B->bases = (BandAff*)b; B->scal = (uint8_t*)s;
  B->seed = (uint8_t*)m; B->bad = (uint32_t*)((uint8_t*)m + 32); B->verdict = (uint8_t*)m + 48; B->prod = (uint32_t*)((uint8_t*)m + 256);
  B->partial = B->prod + 16 * n;
  mark_secret(ctx, BUF_PB2, 32);                                   // the seed: zeroed when the call returns
  CU(cudaMemcpyAsync(B->seed, seed, 32, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemsetAsync(B->bad, 0, 16, ctx->stream));
  return VRFS_OK;
}
// the MSM of the combination and its identity test: *verdict = 1 iff the sum is the identity and *bad = 0
static vrfs_status te_msm_verdict_dev(vrfs_ctx* ctx, size_t nbases, const BandAff* bases, const uint8_t* scal, const uint32_t* bad, uint8_t* verdict) {
  const MsmPlan p = te_msm_plan((uint32_t)nbases);
  const size_t nbuckets = (size_t)p.windows * p.nb, runs = (size_t)p.windows * (p.nb / TE_MSM_CHUNK);
  void *counts = nullptr, *list = nullptr, *buckets = nullptr, *sums = nullptr;
  // counts | offsets | cursors | big_count (16 words) | big_list (never written: te_msm_plan lists no oversized bucket)
  ST(ensure(ctx, BUF_W1, (nbuckets * 3 + 16 + 2) * sizeof(uint32_t), &counts));
  uint32_t *offsets = (uint32_t*)counts + nbuckets, *cursors = offsets + nbuckets, *big_count = cursors + nbuckets, *big_list = big_count + 16;
  ST(ensure(ctx, BUF_W2, (size_t)p.windows * nbases * sizeof(uint32_t), &list));
  ST(ensure(ctx, BUF_W3, nbuckets * sizeof(BandPt), &buckets));
  ST(ensure(ctx, BUF_SLAB, (runs + (size_t)p.windows) * sizeof(BandPt), &sums));
  CU(cudaMemsetAsync(counts, 0, (nbuckets * 3 + 16) * sizeof(uint32_t), ctx->stream));
  const unsigned tsc = (unsigned)((nbases + 127) / 128);
  k_msm_histogram<<<tsc, 128, 0, ctx->stream>>>(p, scal, (uint32_t*)counts);
  LAUNCHED_AS(ctx, "te_msm_histogram");
  k_msm_scan<<<(unsigned)p.windows, MSM_SCAN_THREADS, 0, ctx->stream>>>(p, (const uint32_t*)counts, offsets, big_list, big_count);
  LAUNCHED_AS(ctx, "te_msm_scan");
  k_msm_scatter<<<tsc, 128, 0, ctx->stream>>>(p, scal, offsets, cursors, (uint32_t*)list);
  LAUNCHED_AS(ctx, "te_msm_scatter");
  k_te_msm_accumulate<<<(unsigned)((nbuckets * p.tpb + 127) / 128), 128, 0, ctx->stream>>>(p, bases, (const uint32_t*)counts, offsets, (const uint32_t*)list, (BandPt*)buckets);
  LAUNCHED_AS(ctx, "te_msm_accumulate");
  k_te_msm_chunks<<<(unsigned)((runs + 127) / 128), 128, 0, ctx->stream>>>(p, (const BandPt*)buckets, (BandPt*)sums);
  LAUNCHED_AS(ctx, "te_msm_chunks");
  BandPt* wsum = (BandPt*)sums + runs;
  k_te_msm_window_sum<<<(unsigned)p.windows, TE_MSM_WSUM_THREADS, 0, ctx->stream>>>(p, (const BandPt*)sums, wsum);
  LAUNCHED_AS(ctx, "te_msm_window_sum");
  k_te_msm_final<<<1, 32, 0, ctx->stream>>>(p, wsum, bad, verdict);
  LAUNCHED_AS(ctx, "te_msm_final");
  return VRFS_OK;
}
// after the prep kernels of all items: scalars of G and B, the MSM, and the verdict back to the host (synchronous)
static vrfs_status ped_batch_verdict(vrfs_ctx* ctx, size_t n, const PedBatch& B, uint8_t* out_all_ok) {
  const unsigned blocks = (unsigned)std::min((size_t)PED_BATCH_SUM_BLOCKS, (n + 255) / 256);
  k_pedersen_batch_sum<<<blocks, 256, 0, ctx->stream>>>((uint32_t)n, B.prod, B.partial, 0, 0u, nullptr, nullptr);
  LAUNCHED_AS(ctx, "pedersen_batch_sum");
  k_pedersen_batch_sum<<<1, 256, 0, ctx->stream>>>(blocks, B.partial, nullptr, 1, (uint32_t)n, B.bases, B.scal);
  LAUNCHED_AS(ctx, "pedersen_batch_sum_final");
  ST(te_msm_verdict_dev(ctx, PED_BATCH_NP * n + 2, B.bases, B.scal, B.bad, B.verdict));
  ST(copy_out(ctx, out_all_ok, B.verdict, 1));
  return finish_call(ctx);
}
static void ped_batch_all_ok(size_t n, uint8_t* out_ok, uint8_t* out_status) {
  if (out_ok) memset(out_ok, 1, n);
  if (out_status) memset(out_status, VRFS_ITEM_OK, n);
}

extern "C" vrfs_status vrfs_pedersen_batch_verify(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof,
                                                  const uint8_t* ad, const uint64_t* ad_off, const uint8_t* seed, uint8_t* out_all_ok, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (!seed || !out_all_ok || (n && (!input || !output || !proof))) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  *out_all_ok = n == 0;
  if (n == 0) return VRFS_OK;
  ST(ped_batch_begin(ctx, suite, n));
  typedef BandSuite S;
  const uint8_t* d_ad; const uint64_t* d_off;
  // in pieces: the prep kernel of piece k runs while piece k + 1 (384 B per item) is still on its way
  HostIn in[3] = {{BUF_IN0, input, 64, false, nullptr}, {BUF_IN1, output, 64, false, nullptr}, {BUF_IN2, proof, 256, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 3, &pc, VRFS_HOST_PIECES));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  PedBatch B;
  ST(ped_batch_alloc(ctx, n, seed, &B));
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    k_pedersen_batch_prep<S, true><<<item_blocks(m), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)m, (uint32_t)o, in[0].dev + o * 64, in[1].dev + o * 64, in[2].dev + o * 256,
                                                                                     d_ad, d_off ? d_off + o : nullptr, nullptr, nullptr, B.seed, B.bases, B.scal, B.prod, B.bad);
    LAUNCHED_AS(ctx, "pedersen_batch_prep");
  }
  ST(ped_batch_verdict(ctx, n, B, out_all_ok));
  if (*out_all_ok) { ped_batch_all_ok(n, out_ok, out_status); return VRFS_OK; }
  if (!out_ok && !out_status) return VRFS_OK;
  // rejected: the per-item verifier over the inputs already on the device (exactly what vrfs_pedersen_verify_batch returns)
  uint8_t *d_ok, *d_st = nullptr;
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  ST(pedersen_verify_dev<S>(ctx, n, in[0].dev, in[1].dev, in[2].dev, d_ad, d_off, d_ok, d_st));
  if (out_ok) ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_pedersen_batch_verify_wire(vrfs_ctx* ctx, vrfs_suite suite, size_t n, const uint8_t* data, const uint64_t* data_off, const uint8_t* sig,
                                                       const uint8_t* ad, const uint64_t* ad_off, const uint8_t* seed, uint8_t* out_all_ok, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (!seed || !out_all_ok || (n && (!data_off || !sig))) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  *out_all_ok = n == 0;
  if (n == 0) return VRFS_OK;
  ST(ped_batch_begin(ctx, suite, n));
  typedef BandSuite S;
  const size_t sl = (size_t)vrfs_suite_pedersen_signature_len(suite);
  const uint8_t *d_sig, *d_ad, *d_data; const uint64_t *d_off, *d_doff;
  uint8_t *d_in, *d_out, *d_pr, *d_flags;
  ST(stage_in(ctx, BUF_X1, sig, n * sl, &d_sig));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_var(ctx, BUF_X2, BUF_X3, n, data, data_off, &d_data, &d_doff));
  ST(stage_out(ctx, BUF_IN0, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN1, n * 64, &d_out)); ST(stage_out(ctx, BUF_IN2, n * 256, &d_pr));
  ST(stage_out(ctx, BUF_X4, 6 * n, &d_flags));
  ST((pedersen_wire_decode_dev<S, 4>(ctx, n, d_data, d_doff, d_sig, d_in, d_out, d_pr, d_flags)));
  PedBatch B;
  ST(ped_batch_alloc(ctx, n, seed, &B));
  // the decoder has subgroup-checked the output and the proof's points, and hash-to-curve lands in the subgroup
  k_pedersen_batch_prep<S, false><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, 0u, d_in, d_out, d_pr, d_ad, d_off, d_flags + 4 * n, d_flags + 5 * n,
                                                                                    B.seed, B.bases, B.scal, B.prod, B.bad);
  LAUNCHED_AS(ctx, "pedersen_batch_prep_wire");
  ST(ped_batch_verdict(ctx, n, B, out_all_ok));
  if (*out_all_ok) { ped_batch_all_ok(n, out_ok, out_status); return VRFS_OK; }
  if (!out_ok && !out_status) return VRFS_OK;
  uint8_t *d_ok, *d_st = nullptr;
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  ST((pedersen_wire_verdicts_dev<S, 4>(ctx, n, d_ad, d_off, d_in, d_out, d_pr, d_flags, d_ok, d_st)));
  if (out_ok) ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}

// =================================================================================================
// ring commitment MSM (K12)
// =================================================================================================
// prepared bases (vrfs_msm_g1_prepare): the RingContext analogue - the SRS is fixed, so 2^(c w) P_i is computed once
struct vrfs_msm_bases {
  vrfs_ctx* ctx;    // nullptr once the context was destroyed first (the table is gone; release only frees this record)
  size_t n;
  MsmPlan plan;     // the plan that sized and filled Q (window bits c, windows); per-call plans keep its c
  int tpb_hint;     // 0 = automatic
  void* Q;          // windows * n affine points (96 B each; identity = zeros)
  void* T;          // table mode (msm.cuh "TABLE mode"): 32 * n * 128 affine multiples, or nullptr (bucket mode)
};
#ifndef VRFS_TABLE_TERMS
#define VRFS_TABLE_TERMS 4       // table entries per thread of k_msm_table_sum (sweep: profiles/r3e_table_shapes.log)
#endif
#ifndef VRFS_TABLE_BLOCKS_PER_SM
#define VRFS_TABLE_BLOCKS_PER_SM 2
#endif
#ifndef VRFS_MSM_TABLE_MAX_N
#define VRFS_MSM_TABLE_MAX_N 16384  // SRS sizes up to this get the multiples table by default (393 KB per base: 0.8 GB at 2^11, 6.4 GB at 2^14; 3 columns: 2^13 0.50 vs 0.67 ms, 2^14 0.83 vs 0.93 ms with buckets)
#endif
// the plan of one call on prepared bases: window size and count are the handle's (they fix the layout of Q), only the
// column count (and with it the threads per bucket) is per call
static MsmPlan plan_for(const vrfs_msm_bases* h, int n_columns) {
  return msm_plan((uint32_t)h->n, (uint32_t)n_columns, 1, h->plan.c, h->tpb_hint);
}
// bases: G1Aff[n] (stateless) or the prepared table Q; scalars on the device
static vrfs_status msm_dev(vrfs_ctx* ctx, MsmPlan p, const void* d_bases, const uint8_t* d_scalars, uint8_t* d_out, int out_mode, const PeerArgs* peer = nullptr) {
  const size_t n = p.n, ncol = p.ncol;
  const size_t segs = ncol * p.seg_windows, nbuckets = segs * p.nb, seg_len = n * (p.prepared ? p.windows : 1);
  void *counts = nullptr, *list = nullptr, *buckets = nullptr, *wsum = nullptr;
  // counts | offsets | cursors | big_count (16 words) | slice list of the oversized buckets (2 words per slice) ; partial sums of the slices
  const size_t bigcap = msm_big_capacity(nbuckets, segs * seg_len);
  const size_t w1_words = nbuckets * 3 + 16 + 2 * bigcap;
  ST(ensure(ctx, BUF_W1, w1_words * sizeof(uint32_t) + 16 + bigcap * sizeof(G1Pt), &counts));
  uint32_t *offsets = (uint32_t*)counts + nbuckets, *cursors = offsets + nbuckets, *big_count = cursors + nbuckets, *big_list = big_count + 16;
  G1Pt* bigpart = (G1Pt*)(((uintptr_t)((uint32_t*)counts + w1_words) + 15) & ~(uintptr_t)15);
  ST(ensure(ctx, BUF_W2, segs * seg_len * sizeof(uint32_t), &list));
  ST(ensure(ctx, BUF_W3, nbuckets * sizeof(G1Pt), &buckets));
  // parts[segs * nparts] | row and column sums [segs * (R + H)] | scratch of the weighted sums
  const unsigned nparts = p.rc_h ? 2u : 1u;
  const size_t rc_len = p.rc_h ? (size_t)(p.nb / p.rc_h + p.rc_h) : 0;
  const unsigned wb = (unsigned)msm_wbits(p);                       // results per weighted sum (one per bit of the weights)
  ST(ensure(ctx, BUF_SLAB, (segs * nparts * wb + segs * rc_len + segs) * sizeof(G1Pt), &wsum));
  G1Pt* rc_out = (G1Pt*)wsum + segs * nparts * wb;
  G1Pt* seg_sums = rc_out + segs * rc_len;
  CU(cudaMemsetAsync(counts, 0, (nbuckets * 3 + 16) * sizeof(uint32_t), ctx->stream));
  const unsigned tsc = (unsigned)((n * ncol + 127) / 128);
  k_msm_histogram<<<tsc, 128, 0, ctx->stream>>>(p, d_scalars, (uint32_t*)counts);
  LAUNCHED_AS(ctx, "msm_histogram");
  k_msm_scan<<<(unsigned)segs, MSM_SCAN_THREADS, 0, ctx->stream>>>(p, (const uint32_t*)counts, offsets, big_list, big_count);
  LAUNCHED_AS(ctx, "msm_scan");
  k_msm_scatter<<<tsc, 128, 0, ctx->stream>>>(p, d_scalars, offsets, cursors, (uint32_t*)list);
  LAUNCHED_AS(ctx, "msm_scatter");
  const unsigned bigb = (unsigned)(ctx->sms * 4);
  // Large calls (several resident waves of 4 blocks per SM): the main launch takes the first buckets, the last VRFS_MSM_TAIL_16THS
  // sixteenths run as a second launch with 4 x the threads per bucket on the side stream.  Its tasks are 4 x shorter and start as
  // the main launch drains, so the end of the accumulation is not one long task per idle SM.
  size_t b_main = nbuckets;
  MsmPlan pt = p;
  // (measured, profiles/r3i_msm_tail_ab.log: the stateless mode gains 3-7 % at 2^16 / 2^17 - its (column, window) segments load their
  //  buckets unevenly -, the prepared mode LOSES 4 % at 2^17 - uniform buckets, and the tail's deeper trees cost more than they save)
  if (VRFS_MSM_TAIL_16THS > 0 && !p.prepared && p.tpb * 4 <= 32 && nbuckets * p.tpb > (size_t)ctx->sms * 4 * 128 * 2) {
    b_main = nbuckets / 16 * (16 - VRFS_MSM_TAIL_16THS);
    b_main -= b_main % (128 / p.tpb);                               // whole blocks
    pt.tpb = p.tpb * 4;
  }
  const unsigned ab = (unsigned)((b_main * p.tpb + 127) / 128);
  const unsigned ab_tail = (unsigned)(((nbuckets - b_main) * pt.tpb + 127) / 128);
  const auto accumulate = p.prepared ? k_msm_accumulate<true> : k_msm_accumulate<false>;
  const auto accumulate_big = p.prepared ? k_msm_accumulate_big<true> : k_msm_accumulate_big<false>;
  if (ab_tail) ST(side_fork(ctx));
  accumulate<<<ab, 128, 0, ctx->stream>>>(p, d_bases, (const uint32_t*)counts, offsets, (const uint32_t*)list, (G1Pt*)buckets, (size_t)0, b_main);
  if (ab_tail) {
    accumulate<<<ab_tail, 128, 0, ctx->copy_stream>>>(pt, d_bases, (const uint32_t*)counts, offsets, (const uint32_t*)list, (G1Pt*)buckets, b_main, nbuckets);
    ST(side_join(ctx));
    ctx->launches++;
  }
  LAUNCHED_AS(ctx, "msm_accumulate");
  accumulate_big<<<bigb, MSM_BIG_THREADS, 0, ctx->stream>>>(p, d_bases, (const uint32_t*)counts, offsets, (const uint32_t*)list, big_list, big_count, bigpart);
  LAUNCHED_AS(ctx, "msm_accumulate_big");
  k_msm_big_combine<<<bigb, MSM_BIG_THREADS, 0, ctx->stream>>>(big_list, big_count, bigpart, (G1Pt*)buckets);
  LAUNCHED_AS(ctx, "msm_big_combine");
  if (p.rc_h) {
    k_msm_rc<<<dim3((unsigned)rc_len, (unsigned)segs), 128, 0, ctx->stream>>>(p, (const G1Pt*)buckets, rc_out);
    LAUNCHED_AS(ctx, "msm_rc");
  }
  k_msm_wbits<<<dim3(wb, nparts, (unsigned)segs), 256, 0, ctx->stream>>>(p, p.rc_h ? (const G1Pt*)rc_out : (const G1Pt*)buckets, (G1Pt*)wsum);
  LAUNCHED_AS(ctx, "msm_wsum");
  int final_parts = (int)(nparts * wb);
  const G1Pt* final_in = (const G1Pt*)wsum;
  if (!p.prepared) {                                                // 20 windows per column: add their parts side by side, not inside the Horner chain
    k_msm_sum_parts<<<(unsigned)segs, 32, 0, ctx->stream>>>(final_parts, (const G1Pt*)wsum, seg_sums);
    LAUNCHED_AS(ctx, "msm_sum_parts");
    final_parts = 1; final_in = seg_sums;
  }
  PeerArgs pa = {};
  if (out_mode == 2) { if (!peer) return fail(ctx, VRFS_BAD_ARG, "internal: peer exchange without a peer group"); pa = *peer; }
  k_msm_final2<<<(unsigned)ncol, 32, 0, ctx->stream>>>(p, final_parts, final_in, d_out, out_mode, pa);
  LAUNCHED_AS(ctx, "msm_final");
  return VRFS_OK;
}
// prepared MSM of n_columns scalar columns (device) over a handle: the multiples table when the handle has one, else the buckets
static vrfs_status msm_prepared_dev(vrfs_ctx* ctx, const vrfs_msm_bases* h, int n_columns, int warp_agg, const uint8_t* d_scalars, uint8_t* d_out, int out_mode,
                                    const PeerArgs* peer = nullptr) {
  MsmPlan p = plan_for(h, n_columns);
  p.warp_agg = warp_agg;
  if (!h->T) return msm_dev(ctx, p, h->Q, d_scalars, d_out, out_mode, peer);
  const size_t n = h->n, M = n * MSM_TABLE_WINDOWS;
  // ~8 table entries per thread, at most two blocks per SM and column set (the block trees and the reduction grow with the blocks)
  size_t bpc = (M + 128 * VRFS_TABLE_TERMS - 1) / (128 * VRFS_TABLE_TERMS);
  const size_t cap = (size_t)ctx->sms * VRFS_TABLE_BLOCKS_PER_SM / (size_t)n_columns;
  if (bpc > cap) bpc = cap;
  if (bpc < 1) bpc = 1;
  void* scratch = nullptr;
  ST(ensure(ctx, BUF_SLAB, ((size_t)n_columns * bpc + n_columns) * sizeof(G1Pt), &scratch));
  G1Pt* partials = (G1Pt*)scratch;
  G1Pt* sums = partials + (size_t)n_columns * bpc;
  k_msm_table_sum<<<dim3((unsigned)bpc, (unsigned)n_columns), 128, 0, ctx->stream>>>((uint32_t)n, (const G1Aff*)h->T, d_scalars, partials);
  LAUNCHED_AS(ctx, "msm_table_sum");
  k_msm_table_reduce<<<(unsigned)n_columns, 256, 0, ctx->stream>>>((int)bpc, partials, sums);
  LAUNCHED_AS(ctx, "msm_table_reduce");
  PeerArgs pa = {};
  if (out_mode == 2) { if (!peer) return fail(ctx, VRFS_BAD_ARG, "internal: peer exchange without a peer group"); pa = *peer; }
  k_msm_final2<<<(unsigned)n_columns, 32, 0, ctx->stream>>>(p, 1, sums, d_out, out_mode, pa);
  LAUNCHED_AS(ctx, "msm_final");
  return VRFS_OK;
}
// the stateless MSM over Montgomery affine bases on the device: GLV halves over [P | -phi(P)] (msm.cuh), then the bucket pipeline
static vrfs_status msm_stateless_dev(vrfs_ctx* ctx, size_t n, int ncol, const void* d_aff, const uint8_t* d_scalars, uint8_t* d_out, int out_mode, int window_bits = 0) {
  void *bases2 = nullptr, *scalars2 = nullptr;
  ST(ensure(ctx, BUF_X4, 2 * n * sizeof(G1Aff), &bases2));
  ST(ensure(ctx, BUF_X5, 2 * n * 32 * (size_t)ncol, &scalars2));
  k_msm_glv_split<<<(unsigned)((n * ncol + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, (uint32_t)ncol, (const G1Aff*)d_aff, d_scalars, (G1Aff*)bases2, (uint8_t*)scalars2);
  LAUNCHED_AS(ctx, "msm_glv_split");
  return msm_dev(ctx, msm_plan((uint32_t)(2 * n), (uint32_t)ncol, 0, window_bits, 0, 128), bases2, (const uint8_t*)scalars2, d_out, out_mode);
}
static vrfs_status msm_host(vrfs_ctx* ctx, size_t n, const uint8_t* bases, const uint8_t* scalars, int ncol, uint8_t* out, int out_mode, int window_bits = 0) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (ncol < 1 || ncol > 32) return fail(ctx, VRFS_BAD_ARG, "n_columns must be in 1..32");
  if (!out || (n && (!bases || !scalars))) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  const size_t ob = out_mode ? 144 : 96;
  if (n == 0) {                                   // empty sum = identity
    memset(out, 0, ob * ncol);
    if (out_mode) for (int c = 0; c < ncol; c++) out[ob * c + 48] = 1;   // (0 : 1 : 0)
    return VRFS_OK;
  }
  if (n > (1u << 26)) return fail(ctx, VRFS_BAD_ARG, "MSM size above 2^26 is not supported");
  ST(begin_call(ctx, n));
  const uint8_t *d_b, *d_s; uint8_t* d_o;
  ST(stage_in(ctx, BUF_IN0, bases, n * 96, &d_b)); ST(stage_in(ctx, BUF_IN1, scalars, n * 32 * (size_t)ncol, &d_s));
  ST(stage_out(ctx, BUF_OUT0, ob * ncol, &d_o));
  void* bases_m = nullptr;
  ST(ensure(ctx, BUF_W0, n * sizeof(G1Aff), &bases_m));
  k_msm_prep_bases<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, d_b, (G1Aff*)bases_m);
  LAUNCHED_AS(ctx, "msm_prep_bases");
  ST(msm_stateless_dev(ctx, n, ncol, bases_m, d_s, d_o, out_mode, window_bits));
  ST(copy_out(ctx, out, d_o, ob * ncol));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_msm_g1_bls12_381(vrfs_ctx* ctx, size_t n, const uint8_t* bases, const uint8_t* scalars, int n_columns, uint8_t* out) {
  return msm_host(ctx, n, bases, scalars, n_columns, out, 0);
}
extern "C" vrfs_status vrfs_msm_g1_bls12_381_ex(vrfs_ctx* ctx, size_t n, const uint8_t* bases, const uint8_t* scalars, int n_columns, int window_bits, uint8_t* out) {
  if (ctx && window_bits != 0 && (window_bits < 7 || window_bits > 16)) return fail(ctx, VRFS_BAD_ARG, "window_bits must be 0 (automatic) or 7..16");
  return msm_host(ctx, n, bases, scalars, n_columns, out, 0, window_bits);
}
extern "C" vrfs_status vrfs_msm_g1_partial(vrfs_ctx* ctx, size_t n, const uint8_t* bases, const uint8_t* scalars, int n_columns, uint8_t* out_partial) {
  return msm_host(ctx, n, bases, scalars, n_columns, out_partial, 1);
}
static vrfs_status msm_prepare_impl(vrfs_ctx* ctx, size_t n, const uint8_t* bases, int window_bits, int threads_per_bucket, vrfs_msm_bases** out) {
  if (!ctx || !out) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  *out = nullptr;
  if (n == 0 || !bases) return fail(ctx, VRFS_BAD_ARG, "empty base vector");
  if (n > (1u << 24)) return fail(ctx, VRFS_BAD_ARG, "prepared MSM size above 2^24 is not supported");
  // ceil(256 / c) windows must fit k_msm_prepare's per-thread arrays (MSM_MAX_WINDOWS)
  if (window_bits != 0 && (window_bits < 8 || window_bits > 18)) return fail(ctx, VRFS_BAD_ARG, "window_bits must be 0 (automatic) or 8..18");
  if (threads_per_bucket != 0 && (threads_per_bucket < 1 || threads_per_bucket > 32 || (threads_per_bucket & (threads_per_bucket - 1))))
    return fail(ctx, VRFS_BAD_ARG, "threads_per_bucket must be 0 (automatic) or a power of two <= 32");
  ST(begin_call(ctx, n));
  vrfs_msm_bases* h = new (std::nothrow) vrfs_msm_bases();
  if (!h) return fail(ctx, VRFS_CUDA_ERROR, "out of host memory");
  // no hint and a short SRS: the multiples table (window size 8); a window / thread hint asks for the bucket pipeline
  const bool table_mode = window_bits == 0 && threads_per_bucket == 0 && n <= VRFS_MSM_TABLE_MAX_N;
  if (table_mode) window_bits = MSM_TABLE_C;
  h->ctx = ctx; h->n = n; h->tpb_hint = threads_per_bucket; h->plan = msm_plan((uint32_t)n, 1, 1, window_bits, threads_per_bucket); h->Q = nullptr; h->T = nullptr;
  if (h->plan.windows > MSM_MAX_WINDOWS) { delete h; return fail(ctx, VRFS_BAD_ARG, "internal: %d windows exceed MSM_MAX_WINDOWS", h->plan.windows); }
  cudaError_t e = cudaMalloc(&h->Q, (size_t)h->plan.windows * n * sizeof(G1Aff));
  if (e != cudaSuccess) { delete h; return fail(ctx, VRFS_CUDA_ERROR, "cudaMalloc of the prepared table failed: %s", cudaGetErrorString(e)); }
  if (table_mode) {
    if (h->plan.windows != MSM_TABLE_WINDOWS) { cudaFree(h->Q); delete h; return fail(ctx, VRFS_BAD_ARG, "internal: table mode expects %d windows", MSM_TABLE_WINDOWS); }
    e = cudaMalloc(&h->T, (size_t)MSM_TABLE_WINDOWS * n * MSM_TABLE_D * sizeof(G1Aff));
    if (e != cudaSuccess) { cudaGetLastError(); h->T = nullptr; }          // no room for the table: the bucket pipeline serves the handle
  }
  // a failure below must not leak the table (up to GBs) nor hand out a half-built handle
  auto build = [&]() -> vrfs_status {
    const uint8_t* d_b; void* bases_m = nullptr;
    ST(stage_in(ctx, BUF_IN0, bases, n * 96, &d_b));
    ST(ensure(ctx, BUF_W0, n * sizeof(G1Aff), &bases_m));
    k_msm_prep_bases<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, d_b, (G1Aff*)bases_m);
    LAUNCHED_AS(ctx, "msm_prep_bases");
    k_msm_prepare<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, h->plan.c, h->plan.windows, (const G1Aff*)bases_m, (G1Aff*)h->Q);
    LAUNCHED_AS(ctx, "msm_prepare");
    if (h->T) {
      k_msm_table_build<<<(unsigned)(((size_t)MSM_TABLE_WINDOWS * n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, (const G1Aff*)h->Q, (G1Aff*)h->T);
      LAUNCHED_AS(ctx, "msm_table_build");
    }
    return finish_call(ctx);
  };
  vrfs_status st = build();
  if (st != VRFS_OK) { cudaStreamSynchronize(ctx->stream); cudaFree(h->Q); if (h->T) cudaFree(h->T); delete h; return st; }
  ctx->prepared.push_back(h);
  *out = h;
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_msm_g1_prepare(vrfs_ctx* ctx, size_t n, const uint8_t* bases, vrfs_msm_bases** out) {
  return msm_prepare_impl(ctx, n, bases, 0, 0, out);
}
extern "C" vrfs_status vrfs_msm_g1_prepare_ex(vrfs_ctx* ctx, size_t n, const uint8_t* bases, int window_bits, int threads_per_bucket, vrfs_msm_bases** out) {
  return msm_prepare_impl(ctx, n, bases, window_bits, threads_per_bucket, out);
}
// Handles may be released before or after their context: vrfs_ctx_destroy frees the tables of the handles still alive and
// orphans them (ctx = nullptr); releasing an orphan only frees the record.  (Registry guarded by a global mutex because an
// orphan has no context mutex left to take.)
static std::mutex g_handles_mu;
extern "C" void vrfs_msm_g1_release(vrfs_msm_bases* h) {
  if (!h) return;
  vrfs_ctx* ctx;
  { std::lock_guard<std::mutex> g(g_handles_mu); ctx = h->ctx; }
  if (ctx) {
    CallGuard guard_(ctx, __func__);
    std::lock_guard<std::mutex> g(g_handles_mu);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (h->Q) cudaFree(h->Q);
    if (h->T) cudaFree(h->T);
    auto& v = ctx->prepared;
    v.erase(std::remove(v.begin(), v.end(), h), v.end());
  }
  delete h;
}
static void orphan_prepared(vrfs_ctx* ctx) {      // called by vrfs_ctx_destroy (device set, stream synchronised)
  std::lock_guard<std::mutex> g(g_handles_mu);
  for (vrfs_msm_bases* h : ctx->prepared) { if (h->Q) cudaFree(h->Q); if (h->T) cudaFree(h->T); h->Q = nullptr; h->T = nullptr; h->ctx = nullptr; }
  ctx->prepared.clear();
}
static vrfs_status msm_prepared_host(vrfs_ctx* ctx, const vrfs_msm_bases* h, const uint8_t* scalars, int n_columns, uint8_t* out, int out_mode) {
  if (!ctx || !h || h->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n_columns < 1 || n_columns > 32 || !scalars || !out) return fail(ctx, VRFS_BAD_ARG, "bad argument");
  ST(begin_call(ctx, h->n));
  const size_t ob = out_mode ? 144 : 96;
  const uint8_t* d_s; uint8_t* d_o;
  ST(stage_in(ctx, BUF_IN1, scalars, h->n * 32 * (size_t)n_columns, &d_s));
  ST(stage_out(ctx, BUF_OUT0, ob * n_columns, &d_o));
  ST(msm_prepared_dev(ctx, h, n_columns, 0, d_s, d_o, out_mode));
  ST(copy_out(ctx, out, d_o, ob * n_columns));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_msm_g1_prepared(vrfs_ctx* ctx, const vrfs_msm_bases* h, const uint8_t* scalars, int n_columns, uint8_t* out) {
  return msm_prepared_host(ctx, h, scalars, n_columns, out, 0);
}
extern "C" vrfs_status vrfs_msm_g1_prepared_partial(vrfs_ctx* ctx, const vrfs_msm_bases* h, const uint8_t* scalars, int n_columns, uint8_t* out_partial) {
  return msm_prepared_host(ctx, h, scalars, n_columns, out_partial, 1);
}

// =================================================================================================
// ietf verify against prepared public keys
// =================================================================================================
// A verifier that sees millions of proofs from a few thousand known keys makes Y a fixed base like G: with one table of 8-bit
// windows per key, c*Y is 32 mixed additions (16-17 for a 16-byte challenge), with no doublings, window slab or GLV split.
#define VRFS_MAX_PREPARED_KEYS 65536
struct vrfs_public_keys {
  vrfs_ctx* ctx;          // nullptr once the context was destroyed first (the tables are gone; release only frees this record)
  vrfs_suite suite;
  size_t n_keys;
  void* mem;              // one allocation: tables | rows | key_ok
  const void* tables;     // n_keys x key_table_entries<C>() FixEntry, layout [key][window][entry]
  const uint8_t* rows;    // n_keys x 64: the keys as given, or as decoded (the finish kernel encodes pk from them)
  const uint8_t* key_ok;  // n_keys
  bool from_encodings;    // vrfs_public_keys_prepare_encoded: every key with key_ok = 1 passed the decoder's subgroup check
  bool is_inputs;         // the record of a vrfs_inputs handle
};
// Prepared VRF inputs (vrfs_inputs_prepare) share the record, the build and the lifetime rules of prepared keys: the rows are the
// input points Input::new(data) gave, key_ok is input_ok, and the tables serve s*I as the key tables serve c*Y.
struct vrfs_inputs : vrfs_public_keys {};
static void delete_record(vrfs_public_keys* h) {
  if (h->is_inputs) delete static_cast<vrfs_inputs*>(h); else delete h;
}
// What the rows are made from: affine points; encodings (Codec::point_encode), decoded and subgroup-checked by k_decode_checked;
// or VRF input data, hashed to the curve by data_to_point_dev.  key_ok = the decode or hash-to-curve flag AND the affine key test
// of k_key_table_powers.
enum PrepareFrom { FROM_POINTS, FROM_ENCODINGS, FROM_DATA };
template <class S>
static vrfs_status public_keys_prepare(vrfs_ctx* ctx, vrfs_suite suite, size_t n_keys, const uint8_t* pks, const uint64_t* data_off, PrepareFrom from,
                                       uint8_t* out_key_ok, uint8_t* out_rows, vrfs_public_keys** out) {
  typedef typename S::C C;
  typedef typename Grp<C>::FixEntry E;
  const size_t tbytes = n_keys * key_table_entries<C>() * sizeof(E);
  vrfs_public_keys* h = from == FROM_DATA ? new (std::nothrow) vrfs_inputs() : new (std::nothrow) vrfs_public_keys();
  if (!h) return fail(ctx, VRFS_CUDA_ERROR, "out of host memory");
  h->ctx = ctx; h->suite = suite; h->n_keys = n_keys; h->from_encodings = from == FROM_ENCODINGS; h->is_inputs = from == FROM_DATA;
  cudaError_t e = cudaMalloc(&h->mem, tbytes + n_keys * 65);
  if (e != cudaSuccess) {
    cudaGetLastError(); delete_record(h);
    return fail(ctx, VRFS_CUDA_ERROR, "cudaMalloc of %zu bytes of key tables failed: %s", tbytes + n_keys * 65, cudaGetErrorString(e));
  }
  h->tables = h->mem; h->rows = (const uint8_t*)h->mem + tbytes; h->key_ok = h->rows + n_keys * 64;
  // a failure below must not leak the tables nor hand out a half-built handle
  auto build = [&]() -> vrfs_status {
    const uint8_t* d_pk;
    uint8_t* d_dec_ok = nullptr;
    if (from == FROM_ENCODINGS) {
      const uint8_t* d_enc; uint8_t* d_dec;
      ST(stage_in(ctx, BUF_X0, pks, n_keys * S::ENC_LEN, &d_enc));
      ST(stage_out(ctx, BUF_IN0, n_keys * 64, &d_dec)); ST(stage_out(ctx, BUF_X4, n_keys, &d_dec_ok));
      ST(decode_checked_launch<S>(ctx, n_keys, d_enc, S::ENC_LEN, d_dec, nullptr, 0, nullptr, d_dec_ok));
      d_pk = d_dec;
    } else if (from == FROM_DATA) {   // staged like the data of vrfs_ietf_verify_wire_batch
      const uint8_t* d_data; const uint64_t* d_doff; uint8_t* d_pts;
      ST(stage_var(ctx, BUF_X2, BUF_X3, n_keys, pks, data_off, &d_data, &d_doff));
      ST(stage_out(ctx, BUF_IN0, n_keys * 64, &d_pts)); ST(stage_out(ctx, BUF_X4, n_keys, &d_dec_ok));
      ST(data_to_point_dev<S>(ctx, n_keys, d_data, d_doff, d_pts, d_dec_ok));
      d_pk = d_pts;
    } else {
      ST(stage_in(ctx, BUF_IN0, pks, n_keys * 64, &d_pk));
    }
    k_key_table_powers<C><<<(unsigned)((n_keys + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n_keys, d_pk, (E*)h->mem, (uint8_t*)h->rows, (uint8_t*)h->key_ok);
    LAUNCHED_AS(ctx, "key_table_powers");
    const size_t windows = n_keys * fix_windows<C, KEY_FIX_BITS>();
    k_key_table_windows<C><<<(unsigned)((windows + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n_keys, (E*)h->mem);
    LAUNCHED_AS(ctx, "key_table_windows");
    if (d_dec_ok) {   // key_ok &= decode / hash-to-curve flag.  A failure leaves a zero row, which k_key_table_powers rejects on its own; this does not rely on it
      k_merge_flags<<<item_blocks(n_keys), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n_keys, d_dec_ok, nullptr, (uint8_t*)h->key_ok, nullptr, 0u, nullptr);
      LAUNCHED_AS(ctx, "merge_flags");
    }
    if (out_key_ok) ST(copy_out(ctx, out_key_ok, h->key_ok, n_keys));
    if (out_rows) ST(copy_out(ctx, out_rows, h->rows, n_keys * 64));
    return finish_call(ctx);
  };
  const vrfs_status st = build();
  if (st != VRFS_OK) { cudaStreamSynchronize(ctx->stream); cudaFree(h->mem); delete_record(h); return st; }
  ctx->prepared_keys.push_back(h);
  *out = h;
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_public_keys_prepare(vrfs_ctx* ctx, vrfs_suite suite, size_t n_keys, const uint8_t* pks, uint8_t* out_key_ok, vrfs_public_keys** out) {
  if (!ctx || !out) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  *out = nullptr;
  if (!pks) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (n_keys < 1 || n_keys > VRFS_MAX_PREPARED_KEYS) return fail(ctx, VRFS_BAD_ARG, "n_keys must be in 1..%d", VRFS_MAX_PREPARED_KEYS);
  ST(begin_call(ctx, suite, n_keys));
  return with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return public_keys_prepare<S>(ctx, suite, n_keys, pks, nullptr, FROM_POINTS, out_key_ok, nullptr, out); });
}
extern "C" vrfs_status vrfs_public_keys_prepare_encoded(vrfs_ctx* ctx, vrfs_suite suite, size_t n_keys, const uint8_t* pk_enc, uint8_t* out_key_ok,
                                                        vrfs_public_keys** out) {
  if (!ctx || !out) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  *out = nullptr;
  if (!pk_enc) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (n_keys < 1 || n_keys > VRFS_MAX_PREPARED_KEYS) return fail(ctx, VRFS_BAD_ARG, "n_keys must be in 1..%d", VRFS_MAX_PREPARED_KEYS);
  ST(begin_call(ctx, suite, n_keys));
  return with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S; return public_keys_prepare<S>(ctx, suite, n_keys, pk_enc, nullptr, FROM_ENCODINGS, out_key_ok, nullptr, out); });
}
extern "C" vrfs_status vrfs_inputs_prepare(vrfs_ctx* ctx, vrfs_suite suite, size_t n_inputs, const uint8_t* data, const uint64_t* data_off,
                                           uint8_t* out_input_ok, uint8_t* out_points, vrfs_inputs** out) {
  if (!ctx || !out) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  *out = nullptr;
  if (!data_off) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (n_inputs < 1 || n_inputs > VRFS_MAX_PREPARED_KEYS) return fail(ctx, VRFS_BAD_ARG, "n_inputs must be in 1..%d", VRFS_MAX_PREPARED_KEYS);
  ST(begin_call(ctx, suite, n_inputs));
  vrfs_public_keys* h = nullptr;
  ST(with_suite(ctx, suite, [&](auto S_) { typedef decltype(S_) S;
    return public_keys_prepare<S>(ctx, suite, n_inputs, data, data_off, FROM_DATA, out_input_ok, out_points, &h); }));
  *out = static_cast<vrfs_inputs*>(h);
  return VRFS_OK;
}
// Same lifetime rules as vrfs_msm_bases (vrfs_msm_g1_release): released before or after the context, orphaned by vrfs_ctx_destroy.
extern "C" void vrfs_public_keys_release(vrfs_public_keys* h) {
  if (!h) return;
  vrfs_ctx* ctx;
  { std::lock_guard<std::mutex> g(g_handles_mu); ctx = h->ctx; }
  if (ctx) {
    CallGuard guard_(ctx, __func__);
    std::lock_guard<std::mutex> g(g_handles_mu);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(h->mem);
    auto& v = ctx->prepared_keys;
    v.erase(std::remove(v.begin(), v.end(), h), v.end());
  }
  delete_record(h);
}
extern "C" void vrfs_inputs_release(vrfs_inputs* h) { vrfs_public_keys_release(h); }
static void orphan_public_keys(vrfs_ctx* ctx) {   // called by vrfs_ctx_destroy (device set, stream synchronised)
  std::lock_guard<std::mutex> g(g_handles_mu);
  for (vrfs_public_keys* h : ctx->prepared_keys) { cudaFree(h->mem); h->mem = nullptr; h->ctx = nullptr; }
  ctx->prepared_keys.clear();
}

// U = s*G - c*Y_k (k_lincomb_keyed: both terms fixed-base), V = s*I - c*O as in ietf_verify_dev, the finish kernel of ietf_verify_dev
// on the key rows `pk` with the flags `valid` that the caller's gather left.  Small batches run U on the side stream beside V, like
// ietf_verify_dev.  With prepared inputs `pin`, V = s*I_j - c*O over input input_index[i]'s table (k_lincomb_io); `input` then holds
// the gathered input rows, which the finish kernel encodes.
template <class S>
static vrfs_status ietf_verify_keyed_dev(vrfs_ctx* ctx, const vrfs_public_keys* h, size_t n, const uint32_t* key_index, const uint8_t* pk,
                                         const uint8_t* input, const uint8_t* output, const uint8_t* c, const uint8_t* s, const uint8_t* ad,
                                         const uint64_t* ad_off, uint8_t* valid, uint8_t* out_ok, uint8_t* out_status,
                                         const vrfs_public_keys* pin = nullptr, const uint32_t* input_index = nullptr) {
  typedef typename S::C C;
  void *u = nullptr, *v = nullptr;
  ST(need_tables<S>(ctx));
  ST(ensure(ctx, BUF_W0, n * 96, &u));
  ST(ensure(ctx, BUF_W1, n * 96, &v));
  const bool split = n <= (size_t)ctx->sms * VRFS_SPLIT_ITEMS_PER_SM;
  const uint32_t cbits = S::CLEN < 32 ? 8u * S::CLEN : 0u;
  const KeyedArgs K = {(uint32_t)n, s, c, cbits, key_index, (uint32_t)h->n_keys, ctx->fixtab[S::ID][0], h->tables, (uint32_t*)u};
  if (split) ST(side_fork(ctx));
  k_lincomb_keyed<C><<<(unsigned)((n + KEYED_THREADS - 1) / KEYED_THREADS), KEYED_THREADS, 0, split ? ctx->copy_stream : ctx->stream>>>(K);
  LAUNCHED_AS(ctx, "lincomb_keyed");
  LincombArgs A = {};
  A.n = (uint32_t)n;
  A.valid = valid;
  A.out_xyz = (uint32_t*)v;
  if (pin) {
    IoArgs B = {A, input_index, (uint32_t)pin->n_keys};
    B.L.var[0] = {output, 64, c, 32, 1, cbits};
    B.L.fix[0] = {s, 32, 0, pin->tables};
    ST(launch_lincomb_io<C>(ctx, B));
  } else {
    A.var[0] = {input, 64, s, 32, 0, 0};
    A.var[1] = {output, 64, c, 32, 1, cbits};
    ST((launch_lincomb<C, 2, 0>(ctx, A)));
  }
  if (split) ST(side_join(ctx));
  k_ietf_verify_finish<S><<<(unsigned)((n + 128 * FINISH_K - 1) / (128 * FINISH_K)), 128, 0, ctx->stream>>>((uint32_t)n, pk, input, output, c, (const uint32_t*)u,
                                                                                (const uint32_t*)v, ad, ad_off, valid, out_ok, out_status);
  LAUNCHED_AS(ctx, "ietf_verify_finish");
  return VRFS_OK;
}
// item i's row of the prepared inputs into `rows` (k_gather_keys does this for any row table); flag[i] = 0 for an index out of range
// or an input with input_ok = 0
static vrfs_status gather_inputs(vrfs_ctx* ctx, const vrfs_public_keys* pin, size_t n, const uint32_t* input_index, uint8_t* rows, uint8_t* flag) {
  k_gather_keys<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, input_index, (uint32_t)pin->n_keys, pin->rows, pin->key_ok, rows, flag);
  LAUNCHED_AS(ctx, "gather_inputs");
  return VRFS_OK;
}
// With prepared inputs `pin` the input points are gathered by input_index (`input` is not read) and V comes from their tables.
template <class S>
static vrfs_status ietf_verify_prepared_dev(vrfs_ctx* ctx, const vrfs_public_keys* h, size_t n, const uint32_t* key_index, const uint8_t* input,
                                            const uint8_t* output, const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off,
                                            uint8_t* out_ok, uint8_t* out_status, const vrfs_public_keys* pin = nullptr,
                                            const uint32_t* input_index = nullptr) {
  void *valid = nullptr, *pk = nullptr;
  ST(ensure(ctx, BUF_VALID, n, &valid));
  ST(ensure(ctx, BUF_KEYROWS, n * 64, &pk));
  CU(cudaMemsetAsync(valid, 1, n, ctx->stream));
  k_gather_keys<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, key_index, (uint32_t)h->n_keys, h->rows, h->key_ok, (uint8_t*)pk, (uint8_t*)valid);
  LAUNCHED_AS(ctx, "gather_keys");
  if (pin) {
    void* rows = nullptr;
    ST(ensure(ctx, BUF_INROWS, n * 64, &rows));
    ST(gather_inputs(ctx, pin, n, input_index, (uint8_t*)rows, (uint8_t*)valid));
    input = (const uint8_t*)rows;
  }
  return ietf_verify_keyed_dev<S>(ctx, h, n, key_index, (const uint8_t*)pk, input, output, c, s, ad, ad_off, (uint8_t*)valid, out_ok, out_status, pin,
                                  input_index);
}
// serialised signature + data + key index -> verdict (+ Output::hash of accepted items): ietf_verify_wire_dev with the key taken
// from the prepared set.  k_wire_prepared_unpack stands for the decode, parse and gather kernels; flags = wellformed | h2c ok (2n).
// With prepared inputs `pin` the gather of item i's input row stands for hash-to-curve (`data` is not read): its flag is the h2c
// flag, so a bad input index or an input with input_ok = 0 ends like data without a point.
template <class S>
static vrfs_status ietf_verify_prepared_wire_dev(vrfs_ctx* ctx, const vrfs_public_keys* h, size_t n, const uint32_t* key_index, const uint8_t* data,
                                                 const uint64_t* data_off, const uint8_t* sig, const uint8_t* ad, const uint64_t* ad_off, uint8_t* input,
                                                 uint8_t* output, uint8_t* c, uint8_t* s, uint8_t* flags, uint8_t* out_ok, uint8_t* out_hash, uint8_t* out_status,
                                                 const vrfs_public_keys* pin = nullptr, const uint32_t* input_index = nullptr) {
  void *valid = nullptr, *pk = nullptr;
  ST(ensure(ctx, BUF_VALID, n, &valid));
  ST(ensure(ctx, BUF_KEYROWS, n * 64, &pk));
  k_wire_prepared_unpack<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, key_index, (uint32_t)h->n_keys, h->rows, h->key_ok, sig,
                                                                              (uint8_t*)pk, output, c, s, (uint8_t*)valid, flags);
  LAUNCHED_AS(ctx, "wire_prepared_unpack");
  if (pin) {
    CU(cudaMemsetAsync(flags + n, 1, n, ctx->stream));
    ST(gather_inputs(ctx, pin, n, input_index, input, flags + n));
  } else {
    ST(data_to_point_dev<S>(ctx, n, data, data_off, input, flags + n));
  }
  ST(ietf_verify_keyed_dev<S>(ctx, h, n, key_index, (const uint8_t*)pk, input, output, c, s, ad, ad_off, (uint8_t*)valid, out_ok, out_status, pin,
                              input_index));
  if (out_hash) {
    k_point_to_hash<S><<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, output, out_hash);
    LAUNCHED_AS(ctx, "point_to_hash");
  }
  k_merge_flags<<<item_blocks(n), ITEM_THREADS, 0, ctx->stream>>>((uint32_t)n, flags, flags + n, out_ok, out_hash, (uint32_t)S::HLEN, out_status);
  LAUNCHED_AS(ctx, "merge_flags");
  return VRFS_OK;
}
static vrfs_status check_keys(vrfs_ctx* ctx, const vrfs_public_keys* h) {
  if (!h || h->ctx != ctx) return fail(ctx, VRFS_BAD_ARG, "prepared keys of another (or a destroyed) context");
  if (h->is_inputs) return fail(ctx, VRFS_BAD_ARG, "prepared inputs where prepared keys are expected");
  return VRFS_OK;
}
static vrfs_status check_inputs(vrfs_ctx* ctx, const vrfs_public_keys* keys, const vrfs_inputs* in) {
  ST(check_keys(ctx, keys));
  if (!in || in->ctx != ctx || !in->is_inputs) return fail(ctx, VRFS_BAD_ARG, "prepared inputs of another (or a destroyed) context");
  if (in->suite != keys->suite) return fail(ctx, VRFS_BAD_ARG, "prepared keys and inputs of different suites");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ietf_verify_prepared_batch_dev(vrfs_ctx* ctx, const vrfs_public_keys* keys, size_t n, const uint32_t* key_index,
                                                           const uint8_t* input, const uint8_t* output, const uint8_t* c, const uint8_t* s,
                                                           const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ST(check_keys(ctx, keys));
  if (n == 0) return VRFS_OK;
  if (!key_index || !input || !output || !c || !s || !out_ok || (ad && !ad_off)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (!aligned16(key_index) || !aligned16(input) || !aligned16(output) || !aligned16(c) || !aligned16(s))
    return fail(ctx, VRFS_BAD_ARG, "device buffers must be 16-byte aligned");
  ST(begin_call(ctx, keys->suite, n));
  return with_suite(ctx, keys->suite, [&](auto S_) { typedef decltype(S_) S;
    return ietf_verify_prepared_dev<S>(ctx, keys, n, key_index, input, output, c, s, ad, ad_off, out_ok, out_status); });
}
// host buffers: staged in pieces like vrfs_ietf_verify_batch (ietf_verify_host_enqueue), 4 bytes of key index per item instead of 64 of key
extern "C" vrfs_status vrfs_ietf_verify_prepared_batch(vrfs_ctx* ctx, const vrfs_public_keys* keys, size_t n, const uint32_t* key_index,
                                                       const uint8_t* input, const uint8_t* output, const uint8_t* c, const uint8_t* s,
                                                       const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ST(check_keys(ctx, keys));
  if (n == 0) return VRFS_OK;
  if (!key_index || !input || !output || !c || !s || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, keys->suite, n));
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_ok, *d_st = nullptr;
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  HostIn in[5] = {{BUF_IN0, key_index, 4, false, nullptr}, {BUF_IN1, input, 64, false, nullptr}, {BUF_IN2, output, 64, false, nullptr},
                  {BUF_IN3, c, 32, false, nullptr}, {BUF_IN4, s, 32, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 5, &pc, 2));
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, keys->suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_verify_prepared_dev<S>(ctx, keys, m, (const uint32_t*)in[0].dev + o, in[1].dev + o * 64, in[2].dev + o * 64, in[3].dev + o * 32,
                                         in[4].dev + o * 32, d_ad, d_off ? d_off + o : nullptr, d_ok + o, d_st ? d_st + o : nullptr); }));
  }
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}
// serialised signatures verified against keys prepared from their encodings (vrfs_public_keys_prepare_encoded), the key named by
// index: the results of vrfs_ietf_verify_wire_batch on the gathered encodings.  Staged like that call.
extern "C" vrfs_status vrfs_ietf_verify_prepared_wire_batch(vrfs_ctx* ctx, const vrfs_public_keys* keys, size_t n, const uint32_t* key_index,
                                                            const uint8_t* data, const uint64_t* data_off, const uint8_t* sig, const uint8_t* ad,
                                                            const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_hash, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ST(check_keys(ctx, keys));
  // keys that never passed the decoder's subgroup check: c*Y from the table need not be the wire call's c*Y (header)
  if (!keys->from_encodings) return fail(ctx, VRFS_BAD_ARG, "prepared keys not made from encodings (vrfs_public_keys_prepare_encoded)");
  if (n == 0) return VRFS_OK;
  if (!key_index || !data_off || !sig || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, keys->suite, n));
  const size_t sl = (size_t)vrfs_suite_ietf_signature_len(keys->suite), hl = (size_t)vrfs_suite_hash_len(keys->suite);
  const uint8_t *d_ad, *d_data; const uint64_t *d_off, *d_doff;
  uint8_t *d_in, *d_out, *d_c, *d_s, *d_flags, *d_ok, *d_hash = nullptr, *d_st = nullptr;
  // key indices and signatures on the copy stream in one piece, data and ad on the main stream (see vrfs_ietf_verify_wire_batch)
  HostIn in[2] = {{BUF_X0, key_index, 4, false, nullptr}, {BUF_X1, sig, sl, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 2, &pc, 1));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_var(ctx, BUF_X2, BUF_X3, n, data, data_off, &d_data, &d_doff));
  ST(stage_out(ctx, BUF_IN1, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN2, n * 64, &d_out));
  ST(stage_out(ctx, BUF_IN3, n * 32, &d_c)); ST(stage_out(ctx, BUF_IN4, n * 32, &d_s)); ST(stage_out(ctx, BUF_X4, 2 * n, &d_flags));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_hash) ST(stage_out(ctx, BUF_OUT1, n * hl, &d_hash));
  if (out_status) ST(stage_out(ctx, BUF_X5, n, &d_st));
  HostOut out[3] = {{out_ok, d_ok, 1}, {nullptr, nullptr, 0}, {nullptr, nullptr, 0}};
  int nout = 1;
  if (out_hash) out[nout++] = {out_hash, d_hash, hl};
  if (out_status) out[nout++] = {out_status, d_st, 1};
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, keys->suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_verify_prepared_wire_dev<S>(ctx, keys, m, (const uint32_t*)in[0].dev + o, d_data, d_doff + o, in[1].dev + o * sl, d_ad,
                                              d_off ? d_off + o : nullptr, d_in + o * 64, d_out + o * 64, d_c + o * 32, d_s + o * 32, d_flags + o * 2,
                                              d_ok + o, d_hash ? d_hash + o * hl : nullptr, d_st ? d_st + o : nullptr); }));
    ST(pieces_copy_out(ctx, pc, k, out, nout));
  }
  return finish_call(ctx);
}
// proofs against prepared keys AND prepared inputs, both named by index: item i is vrfs_ietf_verify_prepared_batch with
// input[i] = the point of input input_index[i].  Host form staged in pieces like that call, 136 B per item instead of 196.
extern "C" vrfs_status vrfs_ietf_verify_prepared_io_batch_dev(vrfs_ctx* ctx, const vrfs_public_keys* keys, const vrfs_inputs* inputs, size_t n,
                                                              const uint32_t* key_index, const uint32_t* input_index, const uint8_t* output,
                                                              const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off,
                                                              uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ST(check_inputs(ctx, keys, inputs));
  if (n == 0) return VRFS_OK;
  if (!key_index || !input_index || !output || !c || !s || !out_ok || (ad && !ad_off)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (!aligned16(key_index) || !aligned16(input_index) || !aligned16(output) || !aligned16(c) || !aligned16(s))
    return fail(ctx, VRFS_BAD_ARG, "device buffers must be 16-byte aligned");
  ST(begin_call(ctx, keys->suite, n));
  return with_suite(ctx, keys->suite, [&](auto S_) { typedef decltype(S_) S;
    return ietf_verify_prepared_dev<S>(ctx, keys, n, key_index, nullptr, output, c, s, ad, ad_off, out_ok, out_status, inputs, input_index); });
}
extern "C" vrfs_status vrfs_ietf_verify_prepared_io_batch(vrfs_ctx* ctx, const vrfs_public_keys* keys, const vrfs_inputs* inputs, size_t n,
                                                          const uint32_t* key_index, const uint32_t* input_index, const uint8_t* output,
                                                          const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off,
                                                          uint8_t* out_ok, uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ST(check_inputs(ctx, keys, inputs));
  if (n == 0) return VRFS_OK;
  if (!key_index || !input_index || !output || !c || !s || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, keys->suite, n));
  const uint8_t* d_ad; const uint64_t* d_off; uint8_t *d_ok, *d_st = nullptr;
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_status) ST(stage_out(ctx, BUF_OUT1, n, &d_st));
  HostIn in[5] = {{BUF_IN0, key_index, 4, false, nullptr}, {BUF_IN1, input_index, 4, false, nullptr}, {BUF_IN2, output, 64, false, nullptr},
                  {BUF_IN3, c, 32, false, nullptr}, {BUF_IN4, s, 32, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 5, &pc, 2));
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, keys->suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_verify_prepared_dev<S>(ctx, keys, m, (const uint32_t*)in[0].dev + o, nullptr, in[2].dev + o * 64, in[3].dev + o * 32,
                                         in[4].dev + o * 32, d_ad, d_off ? d_off + o : nullptr, d_ok + o, d_st ? d_st + o : nullptr, inputs,
                                         (const uint32_t*)in[1].dev + o); }));
  }
  ST(copy_out(ctx, out_ok, d_ok, n));
  if (out_status) ST(copy_out(ctx, out_status, d_st, n));
  return finish_call(ctx);
}
// serialised signatures by key index and input index: vrfs_ietf_verify_prepared_wire_batch with data[i] = the data of input
// input_index[i], without hash-to-curve.  Staged like that call, minus the data.
extern "C" vrfs_status vrfs_ietf_verify_prepared_io_wire_batch(vrfs_ctx* ctx, const vrfs_public_keys* keys, const vrfs_inputs* inputs, size_t n,
                                                               const uint32_t* key_index, const uint32_t* input_index, const uint8_t* sig,
                                                               const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_hash,
                                                               uint8_t* out_status) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  ST(check_inputs(ctx, keys, inputs));
  if (!keys->from_encodings) return fail(ctx, VRFS_BAD_ARG, "prepared keys not made from encodings (vrfs_public_keys_prepare_encoded)");
  if (n == 0) return VRFS_OK;
  if (!key_index || !input_index || !sig || !out_ok) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, keys->suite, n));
  const size_t sl = (size_t)vrfs_suite_ietf_signature_len(keys->suite), hl = (size_t)vrfs_suite_hash_len(keys->suite);
  const uint8_t* d_ad; const uint64_t* d_off;
  uint8_t *d_in, *d_out, *d_c, *d_s, *d_flags, *d_ok, *d_hash = nullptr, *d_st = nullptr;
  HostIn in[3] = {{BUF_X0, key_index, 4, false, nullptr}, {BUF_X2, input_index, 4, false, nullptr}, {BUF_X1, sig, sl, false, nullptr}};
  Pieces pc;
  ST(stage_in_pieces(ctx, n, in, 3, &pc, 1));
  ST(stage_ad(ctx, n, ad, ad_off, &d_ad, &d_off));
  ST(stage_out(ctx, BUF_IN1, n * 64, &d_in)); ST(stage_out(ctx, BUF_IN2, n * 64, &d_out));
  ST(stage_out(ctx, BUF_IN3, n * 32, &d_c)); ST(stage_out(ctx, BUF_IN4, n * 32, &d_s)); ST(stage_out(ctx, BUF_X4, 2 * n, &d_flags));
  ST(stage_out(ctx, BUF_OUT0, n, &d_ok));
  if (out_hash) ST(stage_out(ctx, BUF_OUT1, n * hl, &d_hash));
  if (out_status) ST(stage_out(ctx, BUF_X5, n, &d_st));
  HostOut out[3] = {{out_ok, d_ok, 1}, {nullptr, nullptr, 0}, {nullptr, nullptr, 0}};
  int nout = 1;
  if (out_hash) out[nout++] = {out_hash, d_hash, hl};
  if (out_status) out[nout++] = {out_status, d_st, 1};
  for (int k = 0; k < pc.count; k++) {
    const size_t o = pc.cut[k], m = pc.cut[k + 1] - pc.cut[k];
    ST(piece_ready(ctx, k));
    ST(with_suite(ctx, keys->suite, [&](auto S_) { typedef decltype(S_) S;
      return ietf_verify_prepared_wire_dev<S>(ctx, keys, m, (const uint32_t*)in[0].dev + o, nullptr, nullptr, in[2].dev + o * sl, d_ad,
                                              d_off ? d_off + o : nullptr, d_in + o * 64, d_out + o * 64, d_c + o * 32, d_s + o * 32, d_flags + o * 2,
                                              d_ok + o, d_hash ? d_hash + o * hl : nullptr, d_st ? d_st + o : nullptr, inputs,
                                              (const uint32_t*)in[1].dev + o); }));
    ST(pieces_copy_out(ctx, pc, k, out, nout));
  }
  return finish_call(ctx);
}
// =================================================================================================
// ring fixed columns + commitment (SURVEY 8f-2; csrc/ring.cuh)
// =================================================================================================
// evaluations <-> coefficients over the size-2^logn domain, in/out canonical 32-byte LE on the device (may alias)
static vrfs_status ntt_dev(vrfs_ctx* ctx, int logn, uint32_t ncol, int inverse, const uint8_t* d_in, uint8_t* d_out) {
  const size_t n = (size_t)1 << logn, total = n * ncol;
  void *work = nullptr, *tw = nullptr;
  ST(ensure(ctx, BUF_X3, total * sizeof(Fr255), &work));
  ST(ensure(ctx, BUF_X4, (n / 2 + 1) * sizeof(Fr255), &tw));
  k_ntt_twiddles<<<(unsigned)((n / 2 + 1 + 127) / 128), 128, 0, ctx->stream>>>(logn, inverse, (Fr255*)tw);   // n/2 twiddles + the 1/n scale
  LAUNCHED_AS(ctx, "ntt_twiddles");
  k_ntt_load<<<(unsigned)((total + 127) / 128), 128, 0, ctx->stream>>>(logn, ncol, d_in, (Fr255*)work);
  LAUNCHED_AS(ctx, "ntt_load");
  const int fused = logn < NTT_FUSED_LOG ? logn : NTT_FUSED_LOG;
  if (fused > 0) {
    k_ntt_fused<<<(unsigned)(total >> fused), 512, 0, ctx->stream>>>(logn, fused, (const Fr255*)tw, (Fr255*)work);
    LAUNCHED_AS(ctx, "ntt_fused");
  }
  for (int s = fused + 1; s <= logn; s++) {
    k_ntt_stage<<<(unsigned)((total / 2 + 255) / 256), 256, 0, ctx->stream>>>(logn, ncol, s, (const Fr255*)tw, (Fr255*)work);
    LAUNCHED_AS(ctx, "ntt_stage");
  }
  k_ntt_store<<<(unsigned)((total + 127) / 128), 128, 0, ctx->stream>>>(logn, ncol, inverse, (const Fr255*)work, (const Fr255*)tw, d_out);
  LAUNCHED_AS(ctx, "ntt_store");
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_fr_fft_batch(vrfs_ctx* ctx, int log_n, int n_columns, int inverse, const uint8_t* in, uint8_t* out) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (log_n < 0 || log_n > 26 || n_columns < 1 || n_columns > 32 || !in || !out) return fail(ctx, VRFS_BAD_ARG, "bad argument (0 <= log_n <= 26, 1 <= n_columns <= 32)");
  const size_t bytes = ((size_t)n_columns << log_n) * 32;
  ST(begin_call(ctx, (size_t)1 << log_n));
  const uint8_t* d_i; uint8_t* d_o;
  ST(stage_in(ctx, BUF_IN1, in, bytes, &d_i));
  ST(stage_out(ctx, BUF_OUT1, bytes, &d_o));
  ST(ntt_dev(ctx, log_n, (uint32_t)n_columns, inverse != 0, d_i, d_o));
  ST(copy_out(ctx, out, d_o, bytes));
  return finish_call(ctx);
}
// the same transform over BLS12-381 G1 (csrc/g1_fft.cuh): one vector of 2^log_n affine points, in and out 96-byte LE (may alias)
extern "C" vrfs_status vrfs_g1_fft_batch(vrfs_ctx* ctx, int log_n, int inverse, const uint8_t* in, uint8_t* out) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (log_n < 0 || log_n > 24 || !in || !out) return fail(ctx, VRFS_BAD_ARG, "bad argument (0 <= log_n <= 24, non-null buffers)");
  const size_t n = (size_t)1 << log_n;
  ST(begin_call(ctx, n));
  const uint8_t* d_i; uint8_t* d_o; void *work = nullptr, *tw = nullptr;
  ST(stage_in(ctx, BUF_IN0, in, n * 96, &d_i));
  ST(stage_out(ctx, BUF_OUT0, n * 96, &d_o));
  ST(ensure(ctx, BUF_X0, n * sizeof(G1Pt), &work));
  ST(ensure(ctx, BUF_X1, (n / 2 + 1) * sizeof(Fr255), &tw));
  k_ntt_twiddles<<<(unsigned)((n / 2 + 1 + 127) / 128), 128, 0, ctx->stream>>>(log_n, inverse != 0, (Fr255*)tw);   // n/2 twiddles + 1/n
  LAUNCHED_AS(ctx, "ntt_twiddles");
  k_g1_fft_load<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(log_n, d_i, (G1Pt*)work);
  LAUNCHED_AS(ctx, "g1_fft_load");
  for (int s = 1; s <= log_n; s++) {
    k_g1_fft_stage<<<(unsigned)((n / 2 + G1_FFT_STAGE_THREADS - 1) / G1_FFT_STAGE_THREADS), G1_FFT_STAGE_THREADS, 0, ctx->stream>>>(
        log_n, s, (const Fr255*)tw, (G1Pt*)work);
    LAUNCHED_AS(ctx, "g1_fft_stage");
  }
  k_g1_fft_store<<<(unsigned)((n + G1_FFT_STORE_THREADS - 1) / G1_FFT_STORE_THREADS), G1_FFT_STORE_THREADS, 0, ctx->stream>>>(
      log_n, inverse != 0, (const G1Pt*)work, (const Fr255*)tw, d_o);
  LAUNCHED_AS(ctx, "g1_fft_store");
  ST(copy_out(ctx, out, d_o, n * 96));
  return finish_call(ctx);
}
// rows [row_lo, row_lo + n) of the columns; `keys` holds the keys of those rows only (rows row_lo .. min(n_keys, row_lo + n) - 1)
static vrfs_status ring_columns_dev(vrfs_ctx* ctx, size_t n, size_t keyset_part, size_t n_keys, const uint8_t* keys, const uint8_t* padding,
                                    size_t n_tail, const uint8_t* tail, uint8_t** d_cols, size_t row_lo = 0, bool whole_domain = true) {
  if (whole_domain && (n == 0 || (n & (n - 1)) || n > (1u << 26))) return fail(ctx, VRFS_BAD_ARG, "domain size must be a power of two <= 2^26");
  if (n == 0 || row_lo + n > (1u << 26)) return fail(ctx, VRFS_BAD_ARG, "empty or oversized row range");
  if (n_keys > keyset_part || (whole_domain && keyset_part + n_tail > n)) return fail(ctx, VRFS_BAD_ARG, "need n_keys <= keyset_part_size and keyset_part_size + n_tail <= domain size");
  const size_t keys_here = n_keys > row_lo ? std::min(n_keys - row_lo, n) : 0;
  if ((keys_here && !keys) || (n_keys < keyset_part && !padding) || (n_tail && !tail)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  const uint8_t *d_k = nullptr, *d_p = nullptr, *d_t = nullptr;
  ST(stage_in(ctx, BUF_IN0, keys, keys_here * 64, &d_k));
  ST(stage_in(ctx, BUF_IN2, padding, padding ? 64 : 0, &d_p));
  ST(stage_in(ctx, BUF_IN3, tail, n_tail * 64, &d_t));
  void* cols = nullptr;
  ST(ensure(ctx, BUF_IN1, 3 * n * 32, &cols));
  k_ring_columns<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, (uint32_t)row_lo, (uint32_t)keyset_part, (uint32_t)n_keys, d_k, d_p, (uint32_t)n_tail, d_t, (uint8_t*)cols);
  LAUNCHED_AS(ctx, "ring_columns");
  *d_cols = (uint8_t*)cols;
  return VRFS_OK;
}
extern "C" vrfs_status vrfs_ring_fixed_columns(vrfs_ctx* ctx, size_t domain_size, size_t keyset_part_size, size_t n_keys, const uint8_t* keys,
                                               const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_columns) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (!out_columns) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  ST(begin_call(ctx, domain_size));
  uint8_t* d_cols = nullptr;
  ST(ring_columns_dev(ctx, domain_size, keyset_part_size, n_keys, keys, padding, n_tail, tail, &d_cols));
  ST(copy_out(ctx, out_columns, d_cols, 3 * domain_size * 32));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_ring_commit(vrfs_ctx* ctx, const vrfs_msm_bases* srs, int srs_is_lagrange, size_t keyset_part_size, size_t n_keys,
                                        const uint8_t* keys, const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_commitment) {
  if (!ctx || !srs || srs->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (!out_commitment) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  const size_t n = srs->n;
  ST(begin_call(ctx, n));
  uint8_t *d_cols = nullptr, *d_o = nullptr;
  ST(ring_columns_dev(ctx, n, keyset_part_size, n_keys, keys, padding, n_tail, tail, &d_cols));
  if (!srs_is_lagrange) {                          // monomial SRS: commit to the interpolating polynomials
    int logn = 0; while (((size_t)1 << logn) < n) logn++;
    ST(ntt_dev(ctx, logn, 3, 1, d_cols, d_cols));
  }
  ST(stage_out(ctx, BUF_OUT0, 3 * 96, &d_o));
  // (evaluation-form columns repeat the padding point and hold a 0/1 selector: the bucket pipeline aggregates its atomics per warp)
  ST(msm_prepared_dev(ctx, srs, 3, srs_is_lagrange ? 1 : 0, d_cols, d_o, 0));
  ST(copy_out(ctx, out_commitment, d_o, 3 * 96));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_ring_commit_rows_partial(vrfs_ctx* ctx, const vrfs_msm_bases* srs_rows, size_t row_lo, size_t keyset_part_size, size_t n_keys,
                                                     const uint8_t* keys_rows, const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_partial) {
  if (!ctx || !srs_rows || srs_rows->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (!out_partial) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  const size_t n = srs_rows->n;
  ST(begin_call(ctx, n));
  uint8_t *d_cols = nullptr, *d_o = nullptr;
  ST(ring_columns_dev(ctx, n, keyset_part_size, n_keys, keys_rows, padding, n_tail, tail, &d_cols, row_lo, false));
  ST(stage_out(ctx, BUF_OUT0, 3 * 144, &d_o));
  ST(msm_prepared_dev(ctx, srs_rows, 3, 1, d_cols, d_o, 1));
  ST(copy_out(ctx, out_partial, d_o, 3 * 144));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_ring_commit_delta(vrfs_ctx* ctx, const vrfs_msm_bases* srs_lagrange, size_t n_keys, const uint8_t* keys,
                                              const uint8_t* padding, uint8_t* out_delta) {
  if (!ctx || !srs_lagrange || srs_lagrange->ctx != ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  const size_t n = srs_lagrange->n;
  if (!out_delta || !padding || (n_keys && !keys) || n_keys > n) return fail(ctx, VRFS_BAD_ARG, "bad argument (n_keys <= domain size, non-null buffers)");
  ST(begin_call(ctx, n));
  const uint8_t *d_k = nullptr, *d_p = nullptr; uint8_t* d_o = nullptr;
  ST(stage_in(ctx, BUF_IN0, keys, n_keys * 64, &d_k));
  ST(stage_in(ctx, BUF_IN2, padding, 64, &d_p));
  void* cols = nullptr;
  ST(ensure(ctx, BUF_IN1, 2 * n * 32, &cols));
  k_ring_delta_columns<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, (uint32_t)n_keys, d_k, d_p, (uint8_t*)cols);
  LAUNCHED_AS(ctx, "ring_delta_columns");
  ST(stage_out(ctx, BUF_OUT0, 2 * 96, &d_o));
  ST(msm_prepared_dev(ctx, srs_lagrange, 2, 0, (const uint8_t*)cols, d_o, 0));
  ST(copy_out(ctx, out_delta, d_o, 2 * 96));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_g1_compress_batch(vrfs_ctx* ctx, size_t n, const uint8_t* points, uint8_t* out) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n && (!points || !out)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (n == 0) return VRFS_OK;
  ST(begin_call(ctx, n));
  const uint8_t* d_i; uint8_t* d_o;
  ST(stage_in(ctx, BUF_IN0, points, n * 96, &d_i));
  ST(stage_out(ctx, BUF_OUT0, n * 48, &d_o));
  k_g1_compress<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, d_i, d_o);
  LAUNCHED_AS(ctx, "g1_compress");
  ST(copy_out(ctx, out, d_o, n * 48));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_g1_decompress_batch(vrfs_ctx* ctx, size_t n, const uint8_t* enc, int check_subgroup, uint8_t* out_points, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n && (!enc || !out_points || !out_ok)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (n == 0) return VRFS_OK;
  ST(begin_call(ctx, n));
  const uint8_t* d_i; uint8_t *d_o, *d_k;
  ST(stage_in(ctx, BUF_IN0, enc, n * 48, &d_i));
  ST(stage_out(ctx, BUF_OUT0, n * 96, &d_o)); ST(stage_out(ctx, BUF_OUT1, n, &d_k));
  k_g1_decompress<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, d_i, check_subgroup, d_o, d_k);
  LAUNCHED_AS(ctx, "g1_decompress");
  ST(copy_out(ctx, out_points, d_o, n * 96)); ST(copy_out(ctx, out_ok, d_k, n));
  return finish_call(ctx);
}
// self-test / measurement helper: 1/a in BLS12-381 Fq for n canonical 48-byte LE values (0 -> 0); ok[i] = 1 when the
// word-approximation GCD finished on its own (no fallback to the binary Euclid) - the GPU tests require that for every a != 0
__global__ void k_fq381_inv_batch(uint32_t n, const uint8_t* in, uint8_t* out, uint8_t* ok) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t raw[12];
  for (int k = 0; k < 12; k++) raw[k] = k == 0;
  if (i < n) load_le<12>(raw, in + (size_t)48 * i);
  const Fq381 a = to_mont<BlsFq>(raw);
  Fq381 t;
  const bool finished = fq381_inv_bingcd(t, a);
  const Fq381 one_thread = fq381_inv_fast(a);
  // the four-lane form (fq381_inv_coop4) must give the same element: the lanes of a group take their four values in turn
  Fq381 four_lane = one_thread;
  bool four_lane_finished = false;
  for (unsigned turn = 0; turn < 4; turn++) {
    const Fq381 x = fq_shfl(a, (threadIdx.x & 28u) + turn);
    bool fb = false;
    const Fq381 r = fq381_inv_coop4(x, &fb);
    if ((threadIdx.x & 3u) == turn) { four_lane = r; four_lane_finished = !fb; }
  }
  if (i >= n) return;
  ok[i] = (finished && four_lane_finished && four_lane == one_thread) ? 1 : 0;
  from_mont<BlsFq>(raw, four_lane);
  store_le<12>(out + (size_t)48 * i, raw);
}
extern "C" vrfs_status vrfs_fq381_inv_batch(vrfs_ctx* ctx, size_t n, const uint8_t* in, uint8_t* out, uint8_t* out_ok) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n && (!in || !out || !out_ok)) return fail(ctx, VRFS_BAD_ARG, "null buffer");
  if (n == 0) return VRFS_OK;
  ST(begin_call(ctx, n));
  const uint8_t* d_i; uint8_t *d_o, *d_k;
  ST(stage_in(ctx, BUF_IN0, in, n * 48, &d_i));
  ST(stage_out(ctx, BUF_OUT0, n * 48, &d_o)); ST(stage_out(ctx, BUF_OUT1, n, &d_k));
  k_fq381_inv_batch<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((uint32_t)n, d_i, d_o, d_k);
  LAUNCHED_AS(ctx, "fq381_inv_batch");
  ST(copy_out(ctx, out, d_o, n * 48)); ST(copy_out(ctx, out_ok, d_k, n));
  return finish_call(ctx);
}
extern "C" vrfs_status vrfs_g1_sum_partials(vrfs_ctx* ctx, int n_parts, int n_columns, const uint8_t* partials, uint8_t* out) {
  if (!ctx) return VRFS_BAD_ARG;
  CallGuard guard_(ctx, __func__);
  if (n_parts < 1 || n_columns < 1 || n_columns > 32 || !partials || !out) return fail(ctx, VRFS_BAD_ARG, "bad argument");
  ST(begin_call(ctx, 1));
  const uint8_t* d_p; uint8_t* d_o;
  ST(stage_in(ctx, BUF_IN0, partials, (size_t)n_parts * n_columns * 144, &d_p));
  ST(stage_out(ctx, BUF_OUT0, (size_t)96 * n_columns, &d_o));
  k_g1_sum_partials<<<1, 32, 0, ctx->stream>>>(n_parts, n_columns, d_p, d_o);
  LAUNCHED_AS(ctx, "g1_sum_partials");
  ST(copy_out(ctx, out, d_o, (size_t)96 * n_columns));
  return finish_call(ctx);
}

#include "multi_gpu.cuh"
#include "kzg.cuh"
